"""CPU execution of the CUDA sources (tests/emul/cuda_emul.h): the whole device pipeline -- host orchestration in
ss_pipeline.cu and every kernel in ss_kernels.cuh / ss_post.cuh -- compiled with g++ and run thread by thread (CUDA threads
as fibers, warp / block collectives resolved by a scheduler), then checked against the pinned oracle exactly like the GPU
tests do.  This is how kernel logic is verified in the build container, which has no GPU; it is NOT a product path:
the emulated library lives under tests/, is injected only by the fixture below, and is never timed.

What it proves: the statements of the kernels compute the reference's results (bit-exact) for small inputs, for every
code path the GPU tests cover.  What it cannot prove: anything about performance, memory-model races between warps of a
block beyond barrier placement, or sm_100a code generation -- `pytest -m gpu` on the B200 remains the gate."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, free_port, load_golden

EMUL_DIR = os.path.join(ROOT, "tests", "emul")
CSRC = os.path.join(ROOT, "splashsurf_b200", "csrc")


def build_emulated_library() -> str:
    # SS_EMUL_GUARD=1: every device allocation ends in front of an inaccessible page and has no slack, so that any access
    # past a buffer's requested size faults (run the suite once in this mode after touching kernels or buffer sizes)
    guard = bool(os.environ.get("SS_EMUL_GUARD"))
    so = os.path.join(EMUL_DIR, "libsplashsurf_emul_guard.so" if guard else "libsplashsurf_emul.so")
    deps = [os.path.join(EMUL_DIR, "cuda_emul.h")] + [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + \
        [os.path.join(ROOT, "include", "splashsurf_b200.h")]
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("CUDA headers not found")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-g", "-ffp-contract=off", "-fno-fast-math", "-w", "-x", "c++", "-DSS_HOST_EMUL",
                               *(["-DSS_EMUL_GUARD"] if guard else []), "-I" + cuda_inc, "-include", os.path.join(EMUL_DIR, "cuda_emul.h"), "-shared", "-fPIC", "-pthread",
                               "-Wl,-Bsymbolic",      # its cuda* definitions must win over a libcudart that torch may have loaded
                               "-o", so, os.path.join(CSRC, "ss_pipeline.cu")])
    return so


@pytest.fixture(scope="module")
def emu():
    """splashsurf_b200 bound to the emulated library for the duration of this module."""
    import splashsurf_b200 as ss
    so = build_emulated_library()
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


def _parity(oracle_mod, g, o, S=64):
    return oracle_mod.mesh_parity(g.mesh.vertices, g.mesh.triangles, g.vertex_edge_keys, o["vertices"], o["triangles"], o["vertex_keys"], S)


def _check_bit_exact(emu, oracle_mod, p, kw, exact_everywhere=False, tile_batch=None, variant=0, density_variant=0, mc_variant=1):
    ctx = emu.Context()
    try:
        ctx.set_levelset_exact_everywhere(exact_everywhere)
        ctx.set_levelset_variant(variant)
        ctx.set_density_variant(density_variant)
        ctx.set_mc_variant(mc_variant)
        if tile_batch:
            ctx.set_tile_batch(tile_batch)
        g = emu.reconstruct_surface(p, with_debug=True, context=ctx, **kw)
    finally:
        ctx.close()
    o = oracle_mod.reconstruct(p, **kw)
    if o["used_decomposition"]:
        assert np.array_equal(g.subdomains["flat"], o["subdomain_flat"]) and np.array_equal(g.subdomains["count"], o["subdomain_count"])
        assert np.array_equal(g.subdomains["sparse"], o["subdomain_sparse"])
    assert np.array_equal(g.particle_densities, o["particle_densities"])
    m = _parity(oracle_mod, g, o, kw.get("subdomain_num_cubes_per_dim", 64))
    assert m["keys_equal"] and m["triangles_equal"] and m["n_not_bitexact"] == 0, m
    return g, o


@pytest.mark.parametrize("case", ["cfg1_ref", "global_cube_ref", "global_autodisable_ref"])
def test_emulated_matches_reference_fixture(emu, oracle_mod, case):
    """Same assertions as tests/test_gpu_parity.py::test_cuda_matches_reference_fixture (outputs of the reference binary)."""
    gold = load_golden(case)
    g = emu.reconstruct_surface(gold["particles"], with_debug=True, **gold["kwargs"])
    assert np.array_equal(g.grid.aabb.min, gold["grid_min"]) and g.grid.ncells_per_dim == gold["grid_ncells"].tolist()
    assert np.array_equal(g.particle_densities, gold["densities"])
    m = oracle_mod.mesh_parity(g.mesh.vertices, g.mesh.triangles, g.vertex_edge_keys, gold["vertices"], gold["triangles"], gold["keys"],
                               gold["kwargs"].get("subdomain_num_cubes_per_dim", 64))
    assert m["keys_equal"] and m["triangles_equal"], m
    assert m["n_interior_not_bitexact"] == 0 and m["max_abs"] <= 2e-6, m


def _splash(*a):
    from splashsurf_b200 import synthetic as syn
    return syn.splash(*a)


def _cube(*a):
    from splashsurf_b200 import synthetic as syn
    return syn.jittered_cube(*a)


BASE = dict(particle_radius=0.025, smoothing_length=2.0)
SEEDED = [
    ("certify_default", lambda: _cube(12, 0.025, 301), dict(BASE, cube_size=0.5), {}),
    ("exact_everywhere", lambda: _cube(11, 0.025, 302), dict(BASE, cube_size=0.5), dict(exact_everywhere=True)),
    ("scalar_arithmetic", lambda: _splash((10, 10, 10), 2, 0.025, 303), dict(BASE, cube_size=0.6, simd=False), {}),
    ("S20_partial_last_brick", lambda: _splash((10, 10, 10), 2, 0.025, 304),
     dict(BASE, cube_size=0.6, subdomain_num_cubes_per_dim=20, subdomain_grid_auto_disable=False), {}),
    ("S50_partial_last_brick", lambda: _splash((10, 10, 10), 2, 0.025, 305),
     dict(BASE, cube_size=0.6, subdomain_num_cubes_per_dim=50, subdomain_grid_auto_disable=False), {}),
    ("S16_tile_batches_of_2", lambda: _splash((9, 9, 9), 2, 0.025, 306),
     dict(BASE, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False), dict(tile_batch=2)),
    ("l22_c11_S24", lambda: _splash((9, 9, 9), 2, 0.025, 307), dict(particle_radius=0.025, smoothing_length=2.2, cube_size=1.1,
                                                                   subdomain_num_cubes_per_dim=24), {}),
    ("fine_c025", lambda: _splash((6, 6, 6), 1, 0.025, 308), dict(BASE, cube_size=0.25), {}),
    ("global_no_decomposition", lambda: _splash((9, 9, 9), 2, 0.025, 309), dict(BASE, cube_size=0.75, subdomain_grid=False), {}),
    ("threshold_03_density_850", lambda: _cube(10, 0.025, 310), dict(BASE, cube_size=0.5, iso_surface_threshold=0.3, rest_density=850.0), {}),
]


@pytest.mark.parametrize("name,gen,kw,opts", SEEDED, ids=[s[0] for s in SEEDED])
def test_emulated_bit_exact_vs_oracle(emu, oracle_mod, name, gen, kw, opts):
    _check_bit_exact(emu, oracle_mod, gen(), kw, **opts)


@pytest.mark.parametrize("name,gen,kw,opts", [s for s in SEEDED if s[0] != "exact_everywhere"], ids=[s[0] for s in SEEDED if s[0] != "exact_everywhere"])
def test_emulated_split_certification_variant(emu, oracle_mod, name, gen, kw, opts):
    """Level-set variant 1 (ss_certify.cuh: separate certification kernel + exact pass over the failed boxes)."""
    _check_bit_exact(emu, oracle_mod, gen(), kw, variant=1, **opts)


@pytest.mark.parametrize("name,gen,kw,opts", [s for s in SEEDED if s[0] != "exact_everywhere"], ids=[s[0] for s in SEEDED if s[0] != "exact_everywhere"])
def test_emulated_warp_per_brick_certification(emu, oracle_mod, name, gen, kw, opts):
    """Level-set variant 2 (ss_certify.cuh: warp-per-brick certification, bulk-copy staging, packed FP32; the executor runs the
    portable definitions of ss_sm100.cuh)."""
    _check_bit_exact(emu, oracle_mod, gen(), kw, variant=2, **opts)


@pytest.mark.parametrize("n,sigma", [(600, 0.004), (1500, 0.004), (400, 0.02), (260, 0.01), (4500, 0.004)],
                         ids=["oversized_brick_1024_variant", "oversized_brick_4096_variant", "list_overflow", "dense_cluster", "extreme_cluster"])
def test_emulated_warp_per_brick_clustered_particles(emu, oracle_mod, n, sigma):
    """Variant 2 on pathological clustering: more candidates than a warp's slice holds (brick goes to the 4096-candidate variant of
    the exact kernel), more candidates in the support of one sub-box than its list holds, a dense cluster that still fits, and
    more than 4096 candidates around one brick (last resort: k_levelset's selection path)."""
    kw = dict(BASE, cube_size=0.5, subdomain_grid_auto_disable=False)
    _check_bit_exact(emu, oracle_mod, np.random.default_rng(n).normal(0, sigma, (n, 3)).astype(np.float32), kw, variant=2)


@pytest.mark.parametrize("case", ["certify_default", "scalar_arithmetic", "clump_rounds_and_pool_overflow", "clump_oversized_cell", "clumps_in_a_cube"])
def test_emulated_density_kernel_variants(emu, oracle_mod, case):
    """Both density kernels (ss_density.cuh: one warp per h-cell, default; k_density: one thread per particle) against the oracle,
    including the cell-cooperative kernel's escape routes: more than 16 particles of one cell (several rounds), a hit list that
    does not fit the pool (thread-serial routine for that particle), more candidates than the slice holds (whole cell)."""
    kw = dict(BASE, cube_size=0.5, subdomain_grid_auto_disable=False)
    if case in ("certify_default", "scalar_arithmetic"):
        _, gen, kw, _ = [s for s in SEEDED if s[0] == case][0]
        p = gen()
    elif case == "clump_rounds_and_pool_overflow":
        p = np.random.default_rng(7).normal(0, 0.01, (251, 3)).astype(np.float32)      # ~31 particles per cell, ~250 hits each
    elif case == "clump_oversized_cell":
        p = np.random.default_rng(8).normal(0.05, 0.004, (420, 3)).astype(np.float32)  # 420 candidates in one cell
    else:
        rng = np.random.default_rng(9)
        p = np.concatenate([_cube(9, 0.025, 311), rng.normal(0.2, 0.006, (90, 3)).astype(np.float32), rng.normal(0.33, 0.003, (40, 3)).astype(np.float32)])
    for dv in (2, 1, 0):
        _check_bit_exact(emu, oracle_mod, p, kw, variant=2, density_variant=dv)


@pytest.mark.parametrize("name,gen,kw,opts", [s for s in SEEDED if s[0] != "global_no_decomposition"], ids=[s[0] for s in SEEDED if s[0] != "global_no_decomposition"])
def test_emulated_cta_per_brick_passes(emu, oracle_mod, name, gen, kw, opts):
    """The CTA-per-brick marching-cubes / fix-up passes (mc variant 0; the default is the warp-per-brick set of ss_mc.cuh, which
    every other test of this file runs) still produce the reference's mesh."""
    _check_bit_exact(emu, oracle_mod, gen(), kw, variant=2, mc_variant=0, **opts)


def test_emulated_aabb_filter_and_edge_cases(emu, oracle_mod):
    p = _splash((10, 10, 10), 2, 0.025, 320)
    kw = dict(BASE, cube_size=0.6, aabb_min=[-0.05, -0.05, -0.05], aabb_max=[0.4, 1.2, 0.45])
    g, o = _check_bit_exact(emu, oracle_mod, p, kw)
    assert np.array_equal(g.particle_inside_aabb, o["particle_inside_aabb"]) and not g.particle_inside_aabb.all()
    kw = dict(BASE, cube_size=0.5, subdomain_grid_auto_disable=False)
    g = emu.reconstruct_surface(np.zeros((0, 3), np.float32), **kw)                      # empty input
    assert g.mesh.nvertices == 0 and g.mesh.ncells == 0 and g.grid.ncells_per_dim == [64, 64, 64]
    g, _ = _check_bit_exact(emu, oracle_mod, np.array([[0, 0, 0], [3, 3, 3]], np.float32), kw)   # two far-apart particles
    assert g.mesh.nvertices == 252
    # > 512 candidates around one brick: the oversized-candidate path of the level-set kernel
    _check_bit_exact(emu, oracle_mod, np.random.default_rng(1).normal(0, 0.004, (600, 3)).astype(np.float32), kw)
    with pytest.raises(emu.SplashsurfError) as e:
        emu.reconstruct_surface(np.zeros((4, 3), np.float32), particle_radius=0.025, smoothing_length=2.0, cube_size=0.0)
    assert e.value.code == 1


def test_emulated_neighbor_lists_normals_and_tile_tap(emu, oracle_mod):
    p = _splash((9, 9, 9), 2, 0.025, 330)
    kw = dict(BASE, cube_size=0.6)
    o = oracle_mod.reconstruct(p, want_neighbors=True, **kw)
    g = emu.reconstruct_surface(p, global_neighborhood_list=True, **kw)
    off, idx = o["neighbors"]
    assert np.array_equal(g.particle_neighbors.offsets.astype(np.int64), off)
    assert np.array_equal(g.particle_neighbors.indices.astype(np.int64), idx)
    g = emu.reconstruct_surface(p, sph_normals=True, **kw)
    ref = oracle_mod.sph_normals(p, g.particle_densities, g.mesh.vertices, compact_support_radius=0.1,
                                 particle_rest_mass=float(oracle_mod.sph_rest_mass(0.025)))
    assert np.abs(g.normals - ref).max() <= 2e-5
    # the reference's hot-loop fixture (benches/benches/bench_grid_loop.rs:203-262) through ss_levelset_tile_f32
    gl = load_golden("grid_loop_subdomain_33")
    common = dict(global_min=gl["global_min"], cube_size=gl["cell_size"], subdomain_ijk=gl["subdomain_ijk"], subdomain_cubes=64)
    for simd in (True, False):
        t = emu.density_grid_loop(gl["particles"], gl["densities"], compact_support_radius=gl["h"], particle_rest_mass=gl["rest_mass"], simd=simd, **common)
        ref = oracle_mod.levelset_tile(gl["particles"], gl["densities"], subdomain_min=gl["subdomain_min"], h=gl["h"], rest_mass=gl["rest_mass"],
                                       mode=0 if simd else 1, **common)
        assert np.array_equal(t, ref)


# ------------------------------------------------------------------ post-processing (SURVEY 8f) through the same entry points ----
def test_emulated_postprocessing_pipeline(emu, oracle_mod):
    """The GPU post-processing tests (tests/test_zz_gpu_postprocess.py) executed against the emulated library."""
    import test_zz_gpu_postprocess as T
    for name, kw, post in T.CASES:
        T.test_pipeline_postprocessing_matches_oracle(emu, oracle_mod, name, kw, post)
    T.test_pipeline_with_particle_aabb_filters_attributes(emu, oracle_mod)
    T.test_c_abi_smoothing_with_explicit_weights_and_connectivity(emu, oracle_mod)
    T.test_standalone_mesh_functions(emu, oracle_mod)


# ------------------------------------------------------------------ slab partition (multi-GPU entries), ranks run one after another ----
def _virtual_ranks(emu, oracle_mod, x, kw, world, use_callback, force_cuts=None):
    """Runs the per-rank library calls of splashsurf_b200.distributed.Runner._step_multi for `world` slabs in this process
    (the exchange is replaced by selecting each rank's receive set directly) and welds the per-rank meshes like rank 0 does."""
    from splashsurf_b200 import _Grid
    from splashsurf_b200.distributed import make_plan
    ctx = emu.Context()
    L = ctx._L
    p = emu.make_params(**kw)
    corners = np.stack([x.min(axis=0), x.max(axis=0)]).astype(np.float32)
    grid = _Grid()
    assert L.ss_grid_for_reconstruction_f32(ctx._h, corners.ctypes.data, 2, C.byref(p), C.byref(grid)) == 0
    S = int(p.subdomain_num_cubes_per_dim)
    ncells = [int(v) for v in grid.cells_per_dim]
    plan0 = make_plan(ncells, S, float(p.cube_size), float(p.compact_support_radius), None, world)
    ax = plan0.axis
    sub = float(np.float32(np.float32(p.cube_size) * np.float32(S)))
    layer = np.floor((x[:, ax].astype(np.float64) - float(grid.aabb_min[ax])) / sub).astype(np.int64)
    hist = np.bincount(np.clip(layer, 0, plan0.nsub_axis - 1), minlength=plan0.nsub_axis)
    plan = make_plan(ncells, S, float(p.cube_size), float(p.compact_support_radius), hist, world)
    if force_cuts is not None:
        plan.cuts = list(force_cuts)
    recv = []
    for r in range(world):
        lo, hi = plan.recv_range(r)
        recv.append(np.ascontiguousarray(x[(layer >= lo) & (layer < hi)]))          # ascending global order
    # local maxima -> global maximum (the all-reduce MAX of the runner)
    local_max = []
    for r in range(world):
        s = C.c_void_p()
        lo, hi = plan.own(r)
        assert L.ss_reconstruct_partition_f32(ctx._h, recv[r].ctypes.data if len(recv[r]) else None, len(recv[r]), C.byref(p), C.byref(grid),
                                              ax, lo, hi, plan.halo, 0, 1, C.byref(s)) == 0, L.ss_last_error()
        local_max.append(L.ss_surface_max_subdomain_particles(s))
        ctx.free_surface(s)
    gmax = max(local_max)
    # the "stats" protocol gets the same number without any decomposition pre-pass: exact ghost-classifier membership counts of the
    # rank-local particles, summed over the ranks (ss_partition_members_f32; here over contiguous index ranges like Runner.take_local)
    nsd = [(nc + S - 1) // S for nc in ncells]
    members = np.zeros(nsd[0] * nsd[1] * nsd[2], np.int64)
    hist_sum = np.zeros(nsd[ax], np.int64)
    for part in np.array_split(np.arange(len(x)), world):
        xs = np.ascontiguousarray(x[part])
        hist_r, mem_r = np.zeros(nsd[ax], np.uint32), np.zeros(len(members), np.uint32)
        assert L.ss_partition_members_f32(ctx._h, xs.ctypes.data if len(xs) else None, len(xs), C.byref(p), C.byref(grid), ax,
                                          hist_r.ctypes.data, mem_r.ctypes.data) == 0, L.ss_last_error()
        members += mem_r; hist_sum += hist_r
    assert int(members.max()) == gmax, (int(members.max()), gmax)
    assert np.array_equal(hist_sum, hist)
    calls = []
    CB = C.CFUNCTYPE(C.c_uint64, C.c_uint64, C.c_void_p)

    def reduce_cb(local, user):
        calls.append(int(local))
        return gmax
    cb = CB(reduce_cb)
    vs, ks, ts, off = [], [], [], 0
    for r in range(world):
        s = C.c_void_p()
        lo, hi = plan.own(r)
        xp = recv[r].ctypes.data if len(recv[r]) else None
        if use_callback:
            rc = L.ss_reconstruct_partition_cb_f32(ctx._h, xp, len(recv[r]), C.byref(p), C.byref(grid), ax, lo, hi, plan.halo, cb, None, C.byref(s))
        else:
            rc = L.ss_reconstruct_partition_f32(ctx._h, xp, len(recv[r]), C.byref(p), C.byref(grid), ax, lo, hi, plan.halo, gmax, 0, C.byref(s))
        assert rc == 0, L.ss_last_error()
        nv, nt = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s)
        v = np.empty((nv, 3), np.float32); t = np.empty((nt, 3), np.uint32)
        assert L.ss_surface_copy_vertices(s, v.ctypes.data) == 0 and L.ss_surface_copy_triangles_u32(s, t.ctypes.data) == 0
        kp = L.ss_surface_device_vertex_keys(s)
        k = np.frombuffer(C.string_at(kp, nv * 8), dtype=np.uint64).copy() if nv else np.empty(0, np.uint64)
        vs.append(v); ks.append(k); ts.append(t + np.uint32(off)); off += nv
        ctx.free_surface(s)
    if use_callback:
        assert len(calls) == world and sorted(calls) == sorted(int(m) for m in local_max)     # called once per rank, also by empty ranks
    V, K, T = np.ascontiguousarray(np.concatenate(vs)), np.ascontiguousarray(np.concatenate(ks)), np.ascontiguousarray(np.concatenate(ts))
    shift = (42, 22, 2)[ax]
    coord = (K >> np.uint64(shift)) & np.uint64(0xFFFFF)
    cand = np.nonzero(((K & np.uint64(3)) != ax) & np.isin(coord, [c * S for c in plan.cuts[1:-1]]))[0].astype(np.uint32)
    nv_out = C.c_uint64(len(V))
    assert L.ss_weld_meshes(ctx._h, V.ctypes.data, K.ctypes.data, len(V), T.ctypes.data, len(T), cand.ctypes.data if len(cand) else None,
                            len(cand), C.byref(nv_out)) == 0
    ctx.close()
    nvg = int(nv_out.value)
    K = K[:nvg]
    keys4 = np.stack([(K >> np.uint64(42)) & np.uint64(0xFFFFF), (K >> np.uint64(22)) & np.uint64(0xFFFFF), (K >> np.uint64(2)) & np.uint64(0xFFFFF),
                      K & np.uint64(3)], axis=1).astype(np.int64)
    return V[:nvg], T.astype(np.uint64), keys4, plan, [len(a) for a in recv]


@pytest.mark.parametrize("use_callback", [False, True], ids=["two_call", "callback"])
def test_emulated_slab_partition_matches_single_device(emu, oracle_mod, use_callback):
    from splashsurf_b200 import synthetic as syn
    x = syn.dam_break((10, 6, 6), (14, 2, 6), 0.025, 401)                 # long along x: several subdomain layers
    kw = dict(BASE, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False)
    o = oracle_mod.reconstruct(x, **kw)
    for world, cuts in ((2, None), (3, None)):
        v, t, keys, plan, nrecv = _virtual_ranks(emu, oracle_mod, x, kw, world, use_callback, cuts)
        assert plan.nsub_axis >= 3 and all(plan.cuts[r] < plan.cuts[r + 1] for r in range(world)), plan
        m = oracle_mod.mesh_parity(v, t, keys, o["vertices"], o["triangles"], o["vertex_keys"], 16)
        assert m["keys_equal"] and m["triangles_equal"] and m["n_not_bitexact"] == 0, (world, m)


def test_emulated_slab_partition_with_idle_rank(emu, oracle_mod):
    """A rank that owns no subdomain layer and receives no particle still makes every library call (and its max-reduce
    callback), the situation that dead-locked the 8-rank run of round 1."""
    from splashsurf_b200 import synthetic as syn
    x = syn.dam_break((10, 6, 6), (14, 2, 6), 0.025, 402)
    kw = dict(BASE, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False)
    o = oracle_mod.reconstruct(x, **kw)
    nlayers = (int(o["grid"]["ncells"][0]) + 15) // 16
    cuts = [0, nlayers // 2, nlayers // 2, nlayers]                      # rank 1 owns nothing
    for use_callback in (False, True):
        v, t, keys, plan, nrecv = _virtual_ranks(emu, oracle_mod, x, kw, 3, use_callback, cuts)
        assert nrecv[1] == 0
        m = oracle_mod.mesh_parity(v, t, keys, o["vertices"], o["triangles"], o["vertex_keys"], 16)
        assert m["keys_equal"] and m["triangles_equal"] and m["n_not_bitexact"] == 0, m


# ------------------------------------------------------------------ the multi-GPU runner end to end: gloo ranks + CPU executor ----
RUNNER_WORKER = r'''
import ctypes as C, json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SS_ROOT"])
import splashsurf_b200 as ss
from splashsurf_b200 import distributed as ssd, synthetic as syn
ss._LIB = ss._bind(C.CDLL(os.environ["SS_EMUL_SO"]))          # the CUDA sources on the CPU executor (tests only)
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
case = json.loads(os.environ["SS_CASE"])
p_all = getattr(syn, case["gen"])(*[tuple(a) if isinstance(a, list) else a for a in case["args"]])
ctx = ss.Context(0)
runner = ssd.Runner(ctx, ss.make_params(**case["kw"]), world, rank, 0, device="cpu", protocol=case.get("protocol", "stats"))
runner.want_keys = True
x = torch.from_numpy(runner.take_local(p_all))
cuts_seen = []
for it in range(int(case.get("steps", 2))):                     # later steps reuse the pooled buffers; from step 5 on the plan is settled
    out = runner.step(x, copy_out=True)
    cuts_seen.append(list(out["plan"].cuts))
if rank == 0:
    v, t = runner.gathered_mesh(out["nv_global"], out["nt_global"])
    np.savez(os.path.join(os.environ["SS_OUT"], "mesh.npz"), v=v, t=t, k=out["keys_global"].numpy(), cuts=np.asarray(out["plan"].cuts))
json.dump({"recv": out["recv_particles"], "nsub_owned": out["nsub_owned"], "cuts_seen": cuts_seen}, open(os.path.join(os.environ["SS_OUT"], f"rank{rank}.json"), "w"))
ctx.close()
dist.destroy_process_group()
'''


@pytest.mark.parametrize("world,case", [
    (2, dict(gen="dam_break", args=[[10, 6, 6], [14, 2, 6], 0.025, 501],
             kw=dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False))),
    (3, dict(gen="jittered_cube", args=[7, 0.025, 502],     # two subdomain layers for three ranks: one rank stays idle
             kw=dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False))),
    (3, dict(gen="jittered_cube", args=[7, 0.025, 503], protocol="callback",      # one library call, all-reduce from the callback
             kw=dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False))),
    (2, dict(gen="splash", args=[[8, 8, 8], 3, 0.025, 504], protocol="two_call",       # decomposition pre-pass + all-reduce + full call
             kw=dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False))),
    (2, dict(gen="splash", args=[[8, 8, 8], 3, 0.025, 504],                            # same cloud, default protocol: sparse subdomains decided from the statistics
             kw=dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False))),
    (2, dict(gen="dam_break", args=[[10, 6, 6], [14, 2, 6], 0.025, 505], steps=8,     # feedback for four frames, then the best cuts are kept
             kw=dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False))),
], ids=["2_ranks_dam_break", "3_ranks_one_idle", "3_ranks_one_idle_callback", "2_ranks_splash_two_call", "2_ranks_splash_stats", "2_ranks_8_frames_plan_settles"])
def test_emulated_runner_over_gloo(tmp_path, oracle_mod, world, case):
    """splashsurf_b200.distributed.Runner._step_multi as the bench drives it (plan, halo exchange, two library calls, max
    all-reduce, mesh gather + weld), one process per rank over gloo, library = CPU executor; result vs the single-device oracle."""
    import json
    import sys
    from splashsurf_b200 import synthetic as syn
    so = build_emulated_library()
    script = tmp_path / "worker.py"
    script.write_text(RUNNER_WORKER)
    env = dict(os.environ, SS_ROOT=ROOT, SS_OUT=str(tmp_path), SS_EMUL_SO=so, SS_CASE=json.dumps(case), SS_EMUL_THREADS="3", OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), str(script)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    m = np.load(tmp_path / "mesh.npz")
    p_all = getattr(syn, case["gen"])(*[tuple(a) if isinstance(a, list) else a for a in case["args"]])
    o = oracle_mod.reconstruct(p_all, **case["kw"])
    K = m["k"].astype(np.uint64)
    keys4 = np.stack([(K >> np.uint64(42)) & np.uint64(0xFFFFF), (K >> np.uint64(22)) & np.uint64(0xFFFFF), (K >> np.uint64(2)) & np.uint64(0xFFFFF),
                      K & np.uint64(3)], axis=1).astype(np.int64)
    par = oracle_mod.mesh_parity(m["v"], m["t"].astype(np.uint64), keys4, o["vertices"], o["triangles"], o["vertex_keys"], 16)
    assert par["keys_equal"] and par["triangles_equal"] and par["n_not_bitexact"] == 0, par
    ranks = [json.load(open(tmp_path / f"rank{k}.json")) for k in range(world)]
    if world == 3:
        assert min(r_["nsub_owned"] for r_ in ranks) == 0, ranks          # the idle rank really was idle
    assert all(r_["cuts_seen"] == ranks[0]["cuts_seen"] for r_ in ranks)  # every rank took the same plan decisions
    if case.get("steps", 2) >= 7:
        seen = ranks[0]["cuts_seen"]
        assert all(c == seen[4] for c in seen[4:]) and seen[4] in seen[:4], seen   # settled on one of the explored plans


CLI_PARTITION_WORKER = r'''
import ctypes as C, os, sys
sys.path.insert(0, os.environ["SS_ROOT"])
import splashsurf_b200 as ss
ss._LIB = ss._bind(C.CDLL(os.environ["SS_EMUL_SO"]))          # the CUDA sources on the CPU executor (tests only)
from splashsurf_b200 import __main__ as cli
rc = cli.main(sys.argv[1:])
import torch.distributed as dist
if dist.is_initialized():
    dist.destroy_process_group()
sys.exit(rc)
'''


def test_emulated_cli_partitioned_frames_over_gloo(emu, tmp_path):
    """`python -m splashsurf_b200 reconstruct ... --partition=on` under torchrun: every frame of a sequence reconstructed by two processes
    together (splashsurf_b200.distributed.DistributedReconstructor: slab partition, halo exchange, mesh assembled on rank 0) -- the files
    hold the same mesh as the single-process CLI writes (same vertices bit for bit, same triangles; only the numbering differs)."""
    import sys
    from splashsurf_b200 import io, synthetic as syn, __main__ as cli
    frames = tmp_path / "f"
    frames.mkdir()
    for i in (1, 2):
        io.write_particles(str(frames / f"dam_{i}.bgeo"), syn.dam_break((10, 6, 6), (14, 2, 6), 0.025, 600 + i))
    args = ["reconstruct", str(frames / "dam_{}.bgeo"), "-r=0.025", "-l=2.0", "-c=0.75", "--subdomain-cubes", "16", "--particle-aabb-min", "-1", "-1", "-1",
            "--particle-aabb-max", "0.55", "2", "2", "-q"]
    assert cli.main(args + ["--output-dir", str(tmp_path / "one")]) == 0
    script = tmp_path / "worker.py"
    script.write_text(CLI_PARTITION_WORKER)
    env = dict(os.environ, SS_ROOT=ROOT, SS_EMUL_SO=build_emulated_library(), SS_EMUL_THREADS="3", OMP_NUM_THREADS="1", SS_DIST_BACKEND="gloo",
               SS_RUNNER_DEVICE="cpu")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port",
           str(free_port()), str(script), *args, "--partition=on", "--output-dir", str(tmp_path / "two")]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert sorted(os.listdir(tmp_path / "two")) == sorted(os.listdir(tmp_path / "one")) == ["dam_surface_1.vtk", "dam_surface_2.vtk"]
    for f in ("dam_surface_1.vtk", "dam_surface_2.vtk"):
        v1, t1 = io.read_vtk_mesh(str(tmp_path / "one" / f))[:2]
        v2, t2 = io.read_vtk_mesh(str(tmp_path / "two" / f))[:2]
        assert len(v1) == len(v2) > 1000 and len(t1) == len(t2)
        from test_zzzz_reference_datasets import _canonical_mesh
        a, b = _canonical_mesh(v1, t1), _canonical_mesh(v2, t2)
        assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)) and np.array_equal(a[1], b[1])     # the same vertices bit for bit, the same triangles
    # a domain at most 1.2 subdomains wide with auto-disable on (lib.rs:421-440): rank 0 reconstructs the gathered cloud on the global path
    # and holds the mesh (+ SPH normals); same file as the single-process command line
    small = ["reconstruct", str(frames / "dam_1.bgeo"), "-r=0.025", "-l=2.0", "-c=1.5", "--subdomain-grid-auto-disable=off", "--normals=on", "--sph-normals=on",
             "-q", "-o", "small.ply"]
    assert cli.main(small + ["--output-dir", str(tmp_path / "one")]) == 0
    r = subprocess.run(cmd[:cmd.index(str(script)) + 1] + small + ["--partition=on", "--output-dir", str(tmp_path / "two")], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    a, b = io.read_ply_mesh(str(tmp_path / "one" / "small.ply")), io.read_ply_mesh(str(tmp_path / "two" / "small.ply"))
    assert len(a[0]) > 100 and np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[3]["normals"], b[3]["normals"])
    # post-processing is a single-GPU step: refused with a clear message
    r = subprocess.run(cmd + ["--mesh-smoothing-iters=2"], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--partition=on reconstructs without mesh post-processing" in r.stderr


API_EDGE_WORKER = r'''
import ctypes as C, json, os, sys
import numpy as np, torch.distributed as dist
sys.path.insert(0, os.environ["SS_ROOT"])
import splashsurf_b200 as ss
ss._LIB = ss._bind(C.CDLL(os.environ["SS_EMUL_SO"]))
from splashsurf_b200.distributed import DistributedReconstructor
dist.init_process_group("gloo")
rank = dist.get_rank()
rec = DistributedReconstructor(device="cpu", particle_radius=0.025, smoothing_length=2.0, cube_size=0.5, subdomain_grid_auto_disable=False)
out = {}
for name, p in (("empty", np.zeros((0, 3), np.float32)),
                ("one_rank_empty", np.random.default_rng(0).random((300 if rank == 0 else 0, 3)).astype(np.float32) * np.float32(0.4)),
                ("two_particles", np.float32([[0, 0, 0]] if rank == 0 else [[3, 3, 3]]))):
    m = rec(p)
    out[name] = None if m is None else [m.nvertices, m.ncells]
rec.close()
json.dump(out, open(os.path.join(os.environ["SS_OUT"], f"edge{rank}.json"), "w"))
dist.destroy_process_group()
'''


def test_emulated_distributed_reconstructor_edge_cases_over_gloo(emu, tmp_path):
    """DistributedReconstructor with nothing to do on some or all ranks: an empty cloud gives an empty mesh on rank 0 (like the single-device
    call), a rank without particles takes part in every collective, two far-apart particles on two ranks give the single-device mesh."""
    import json
    import sys
    script = tmp_path / "worker.py"
    script.write_text(API_EDGE_WORKER)
    env = dict(os.environ, SS_ROOT=ROOT, SS_OUT=str(tmp_path), SS_EMUL_SO=build_emulated_library(), SS_EMUL_THREADS="3", OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port",
           str(free_port()), str(script)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    r0, r1 = json.load(open(tmp_path / "edge0.json")), json.load(open(tmp_path / "edge1.json"))
    assert r1 == {"empty": None, "one_rank_empty": None, "two_particles": None}
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5, subdomain_grid_auto_disable=False)
    one = emu.reconstruct_surface(np.random.default_rng(0).random((300, 3)).astype(np.float32) * np.float32(0.4), **kw)
    two = emu.reconstruct_surface(np.float32([[0, 0, 0], [3, 3, 3]]), **kw)
    assert r0 == {"empty": [0, 0], "one_rank_empty": [one.mesh.nvertices, one.mesh.ncells], "two_particles": [two.mesh.nvertices, two.mesh.ncells]}


FAIL_WORKER = r'''
import ctypes as C, json, os, sys
import numpy as np, torch, torch.distributed as dist, datetime
sys.path.insert(0, os.environ["SS_ROOT"])
import splashsurf_b200 as ss
from splashsurf_b200 import distributed as ssd, synthetic as syn
ss._LIB = ss._bind(C.CDLL(os.environ["SS_EMUL_SO"]))
dist.init_process_group("gloo", timeout=datetime.timedelta(seconds=60))
rank, world = dist.get_rank(), dist.get_world_size()
p_all = syn.dam_break((10, 6, 6), (14, 2, 6), 0.025, 501)
kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_num_cubes_per_dim=16, subdomain_grid_auto_disable=False)
ctx = ss.Context(0)
runner = ssd.Runner(ctx, ss.make_params(**kw), world, rank, 0, device="cpu", protocol=os.environ["SS_PROTOCOL"])
runner._test_fail_rank = 1
x = torch.from_numpy(runner.take_local(p_all))
try:
    runner.step(x, copy_out=False)
    outcome = "no error"
except RuntimeError as e:
    outcome = "raised: " + str(e)[:120]
json.dump({"outcome": outcome}, open(os.path.join(os.environ["SS_OUT"], f"rank{rank}.json"), "w"))
runner._test_fail_rank = None
out = runner.step(x, copy_out=False)                             # and the group is still usable afterwards
json.dump({"outcome": outcome, "nv_after": int(out["nv"])}, open(os.path.join(os.environ["SS_OUT"], f"rank{rank}.json"), "w"))
ctx.close()
dist.destroy_process_group()
'''


@pytest.mark.parametrize("protocol", ["stats", "callback", "two_call"])
def test_emulated_runner_failure_on_one_rank_raises_everywhere(tmp_path, protocol):
    """A failing library call on one rank must not leave the other ranks blocked in a collective: the max-reduce still happens
    on the failing rank (ss_pipeline.cu: ReduceOnce) and the status all-reduce makes every rank raise."""
    import json
    import sys
    so = build_emulated_library()
    script = tmp_path / "worker.py"
    script.write_text(FAIL_WORKER)
    env = dict(os.environ, SS_ROOT=ROOT, SS_OUT=str(tmp_path), SS_EMUL_SO=so, SS_PROTOCOL=protocol, SS_EMUL_THREADS="3", OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), str(script)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    res = [json.load(open(tmp_path / f"rank{k}.json")) for k in range(2)]
    assert all(x["outcome"].startswith("raised") for x in res), res
    assert "xyz is NULL" in res[1]["outcome"] and "another rank failed" in res[0]["outcome"], res
    assert res[0]["nv_after"] + res[1]["nv_after"] > 0


def test_emulated_large_result_copies_take_the_staged_path(emu, oracle_mod):
    """Result copies larger than four chunks (32 MiB each by default) go device -> page-locked staging -> destination with several
    host threads, and the u32 -> u64 widening of the triangle indices happens on the host; smaller ones are one plain copy.  Both
    must deliver the same bytes: the same surface copied with the default chunk (plain path) and with 64 KiB chunks (staged path)."""
    x = _cube(20, 0.025, 777)
    kw = dict(BASE, cube_size=0.5)
    ctx = emu.Context()
    try:
        p = emu.make_params(**kw)
        xs = np.ascontiguousarray(x)
        s = ctx.reconstruct_raw(xs.ctypes.data, len(xs), p)
        L = ctx._L
        nv, nt = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s)
        got = []
        for chunk in (32 << 20, 64 << 10, 4096 + 4):
            assert L.ss_context_set_copy_chunk_bytes(ctx._h, chunk) == 0
            t32 = np.full((nt, 3), 0xdeadbeef, np.uint32); t64 = np.full((nt, 3), 7, np.uint64); v = np.full((nv, 3), np.nan, np.float32)
            assert L.ss_surface_copy_triangles_u32(s, t32.ctypes.data) == 0 and L.ss_surface_copy_triangles_u64(s, t64.ctypes.data) == 0
            assert L.ss_surface_copy_vertices(s, v.ctypes.data) == 0
            got.append((v, t32, t64))
        assert nt * 12 >= 4 * (64 << 10)                               # the small chunk sizes really took the staged path
        for v, t32, t64 in got[1:]:
            assert np.array_equal(v, got[0][0]) and np.array_equal(t32, got[0][1]) and np.array_equal(t64, got[0][2])
        assert np.array_equal(got[0][1].astype(np.uint64), got[0][2]) and int(got[0][2].max()) == nv - 1
        assert L.ss_context_set_copy_chunk_bytes(ctx._h, 100) != 0     # out of range
        ctx.free_surface(s)
        # the upload of a pageable particle array is staged the same way: 20^3 particles = 96 KB > 4 chunks of 4100 bytes
        assert L.ss_context_set_copy_chunk_bytes(ctx._h, 4096 + 4) == 0
        g = emu.reconstruct_surface(x, context=ctx, **kw)
        o = oracle_mod.reconstruct(x, **kw)
        assert np.array_equal(g.particle_densities, o["particle_densities"]) and g.mesh.nvertices == len(o["vertices"])
    finally:
        ctx.close()


def test_emulated_sph_interpolator_at_arbitrary_points(emu, oracle_mod, reference_output):
    """pysplashsurf.SphInterpolator on the CPU executor: same checks as the GPU-marked test (oracle restatements + the wheel's class)."""
    from test_zzzz_reference_datasets import check_sph_interpolator
    check_sph_interpolator(emu, oracle_mod, reference_output)


def test_emulated_neighborhood_search_stand_alone(emu, oracle_mod, reference_output):
    """pysplashsurf.neighborhood_search_spatial_hashing_parallel on the CPU executor: same checks as the GPU-marked test."""
    from test_zzzz_reference_datasets import check_neighborhood_search
    check_neighborhood_search(emu, oracle_mod, reference_output)


def test_emulated_marching_cubes_on_a_dense_array(emu, oracle_mod, reference_output):
    """pysplashsurf.marching_cubes on the CPU executor: same checks as the GPU-marked test (one-cell KAT, sphere SDF, the wheel's meshes)."""
    from test_zzzz_reference_datasets import check_marching_cubes
    check_marching_cubes(emu, oracle_mod, reference_output)


def test_emulated_cli_sequence_equals_library_calls(emu, tmp_path):
    """The GPU-marked command-line test on the CPU executor."""
    from test_zzzz_reference_datasets import check_cli_sequence
    check_cli_sequence(emu, tmp_path)


def test_emulated_reference_python_tests(emu, tmp_path, oracle_mod):
    """pysplashsurf/tests/*.py against `import splashsurf_b200 as pysplashsurf` on the CPU executor (tests/test_zzzzz_pysplashsurf_tests.py)."""
    from test_zzzzz_pysplashsurf_tests import run_all
    run_all(emu, tmp_path, oracle_mod)


def test_emulated_cli_with_postprocessing(emu, tmp_path):
    """`python -m splashsurf_b200 reconstruct` with the reference CLI's post-processing switches (clean-up, decimation, smoothing, normals,
    mesh checks, quads) -- control flow of the thin harness on the CPU executor."""
    from splashsurf_b200 import io, __main__ as cli
    p = _splash((8, 8, 8), 2, 0.025, 3)
    src = str(tmp_path / "in.xyz")
    io.write_xyz(src, p)
    base = ["reconstruct", src, "-r", "0.025", "-l", "2.0", "-c", "0.75"]
    assert cli.main(base + ["-o", str(tmp_path / "a.obj")]) == 0
    v0, t0 = io.read_obj(str(tmp_path / "a.obj"))[:2]
    assert cli.main(base + ["--mesh-cleanup", "on", "--decimate-barnacles", "on", "--mesh-smoothing-iters", "5", "--mesh-smoothing-weights", "on",
                            "--normals", "on", "--sph-normals", "on", "--check-mesh", "on", "-o", str(tmp_path / "b.obj")]) == 0
    v1, t1 = io.read_obj(str(tmp_path / "b.obj"))[:2]
    assert 0 < len(v1) < len(v0) and 0 < len(t1) < len(t0)
    assert cli.main(base + ["--generate-quads", "on", "-o", str(tmp_path / "c.npz")]) == 0
    z = np.load(tmp_path / "c.npz")
    assert len(z["quads"]) > 0 and len(z["triangles"]) + 2 * len(z["quads"]) == len(t0)
    # output files as the reference CLI writes them: attributes travel in .vtk / .ply, quads in every format; smoothing switches the
    # clean-up on unless told otherwise (reconstruct.rs:200-213)
    sm = ["--mesh-smoothing-iters=2", "--mesh-smoothing-weights=on", "--output-smoothing-weights=on", "--normals=on"]
    assert cli.main(base + sm + ["-o", str(tmp_path / "d.vtk")]) == 0
    assert cli.main(base + sm + ["-o", str(tmp_path / "d.ply")]) == 0
    assert cli.main(base + sm + ["--mesh-cleanup=off", "-o", str(tmp_path / "e.ply")]) == 0
    vd, td, qd, pa, ca = io.read_vtk_mesh(str(tmp_path / "d.vtk"))
    vp, tp, qp, pp = io.read_ply_mesh(str(tmp_path / "d.ply"))
    assert list(pa) == ["wnn", "sw", "normals"] == list(pp) and ca == {} and np.array_equal(vd, vp) and np.array_equal(td, tp)
    assert all(np.array_equal(pa[k], pp[k]) for k in pa) and pa["normals"].shape == (len(vd), 3)
    assert len(vd) < len(io.read_ply_mesh(str(tmp_path / "e.ply"))[0]) == len(v0)          # the clean-up ran by default
    assert cli.main(base + ["--generate-quads=on", "--normals=on", "-o", str(tmp_path / "q.vtk")]) == 0
    vq, tq, qq, paq, _ = io.read_vtk_mesh(str(tmp_path / "q.vtk"))
    assert np.array_equal(tq, z["triangles"]) and np.array_equal(qq, z["quads"]) and list(paq) == ["normals"]


def test_emulated_cli_frame_sequence_beside_reference_cli(emu, oracle_mod, tmp_path, monkeypatch):
    """File sequences like the reference CLI (reconstruct.rs:700-963): "{}" in the input name, -s / -e, default output names, --output-dir,
    raw_ meshes, the particle AABB, bgeo / json / vtk inputs -- same files as the REFERENCE CLI writes for the same command line (names,
    sizes, triangle sets after matching vertices by position); frames sharded over processes (--shard / RANK, WORLD_SIZE) give the same files."""
    import subprocess, sys
    from scipy.spatial import cKDTree
    from splashsurf_b200 import io, __main__ as cli
    frames = tmp_path / "frames"
    frames.mkdir()
    for i, ext in ((2, "bgeo"), (9, "bgeo"), (10, "bgeo"), (11, "bgeo"), (30, "bgeo")):
        io.write_particles(str(frames / f"fluid_{i}_x.{ext}"), _splash((6, 6, 6), 1, 0.025, 40 + i))
    io.write_particles(str(frames / "other_3.bgeo"), _splash((5, 5, 5), 1, 0.025, 1))
    (frames / "fluid__x.bgeo").write_bytes(b"not a frame: no digits")
    common = ["-r=0.025", "-l=2.0", "-c=0.75", "-s", "9", "-e", "11", "--particle-aabb-min", "-1", "-1", "-1", "--particle-aabb-max", "0.2", "2", "2",
              "--output-raw-mesh=on", "--mesh-smoothing-iters=1", "--mesh-cleanup=off", "--normals=on"]
    pattern = str(frames / "fluid_{}_x.bgeo")
    ours, theirs = tmp_path / "ours", tmp_path / "theirs"
    assert cli.main(["reconstruct", pattern, *common, "--output-dir", str(ours), "-q"]) == 0
    expect = sorted(f"{pre}fluid_surface_{i}_x.vtk" for i in (9, 10, 11) for pre in ("", "raw_"))
    assert sorted(os.listdir(ours)) == expect
    # two processes taking every second frame (the device version of --mt-files): same files
    sharded = tmp_path / "sharded"
    assert cli.main(["reconstruct", pattern, *common, "--output-dir", str(sharded), "-q", "--shard", "0/2"]) == 0
    assert sorted(os.listdir(sharded)) == sorted(f"{pre}fluid_surface_{i}_x.vtk" for i in (9, 11) for pre in ("", "raw_"))
    monkeypatch.setenv("RANK", "1"); monkeypatch.setenv("WORLD_SIZE", "2"); monkeypatch.setenv("LOCAL_RANK", "0")
    assert cli.main(["reconstruct", pattern, *common, "--output-dir", str(sharded), "-q"]) == 0
    monkeypatch.delenv("RANK"); monkeypatch.delenv("WORLD_SIZE"); monkeypatch.delenv("LOCAL_RANK")
    assert sorted(os.listdir(sharded)) == expect
    assert all(open(ours / f, "rb").read() == open(sharded / f, "rb").read() for f in expect)
    # explicit output pattern; a pattern without "{}" is refused; inverted ranges are refused
    assert cli.main(["reconstruct", pattern, *common[:3], "-o", "m_{}.ply", "--output-dir", str(tmp_path / "pat"), "-e", "2", "-q"]) == 0
    assert os.listdir(tmp_path / "pat") == ["m_2.ply"]
    with pytest.raises(ValueError, match="does not contain a place holder"):
        cli.main(["reconstruct", pattern, *common[:3], "-o", "m.ply"])
    with pytest.raises(ValueError, match='Invalid input sequence range: "5 to 3"'):
        cli.main(["reconstruct", pattern, *common[:3], "-s", "5", "-e", "3"])
    with pytest.raises(ValueError, match="Input file does not exist"):
        cli.main(["reconstruct", str(frames / "nope.bgeo"), *common[:3]])
    with pytest.raises(ValueError, match="particle AABB is degenerate"):
        cli.main(["reconstruct", pattern, *common[:3], "--particle-aabb-min", "0", "0", "0", "--particle-aabb-max", "1", "0", "1"])
    # a single file without -o: "<stem>_surface.vtk" in the working directory
    monkeypatch.chdir(tmp_path)
    assert cli.main(["reconstruct", str(frames / "other_3.bgeo"), *common[:3], "-q"]) == 0
    assert os.path.isfile(tmp_path / "other_3_surface.vtk")
    if not oracle_mod.reference_available():
        return
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "import sys; sys.path.insert(0, %r); import oracle; oracle.reference().run_splashsurf(['splashsurf'] + sys.argv[1:])" % root
    subprocess.check_call([sys.executable, "-c", code, "reconstruct", pattern, *common, "--output-dir", str(theirs), "-q"])
    assert sorted(os.listdir(theirs)) == expect
    for f in expect:
        assert os.path.getsize(theirs / f) == os.path.getsize(ours / f), f
        v1, t1, _, a1, _ = io.read_vtk_mesh(str(theirs / f))
        v2, t2, _, a2, _ = io.read_vtk_mesh(str(ours / f))
        assert len(v1) == len(v2) > 500 and list(a1) == list(a2) == ([] if f.startswith("raw_") else ["normals"])
        d, idx = cKDTree(v2).query(v1)
        assert d.max() < 2e-6 and len(np.unique(idx)) == len(v1)
        assert set(map(tuple, np.sort(idx[t1], axis=1))) == set(map(tuple, np.sort(t2.astype(np.int64), axis=1)))
        assert v1[:, 0].max() < 0.35                      # the particle AABB cut the cloud


def test_emulated_cli_end_to_end_against_reference_cli_with_attributes(emu, oracle_mod, tmp_path, reference_output):
    """The whole harness path on a reference fixture (SPlisHSPlasH VTK with `id` and `velocity` point data, tests/golden/reference_data):
    particle + attribute readers, clean-up (on by default with smoothing), weighted smoothing, normals, SPH interpolation of both
    attributes (`-a`), PLY writer -- beside the REFERENCE CLI with the same command line.  Same file size, same attribute order, same
    counts; a fixed sample of the reference's vertices (with their attribute values) and of its triangles is stored
    (tests/golden/bunny_cli_ref.npz): the vertices are matched by position (the reference's vertex order is not fixed), every sampled
    triangle is one of ours, values within the f32 summation-order tolerance of DESIGN 3a."""
    import subprocess, sys
    from scipy.spatial import cKDTree
    from conftest import GOLDEN, load_golden
    from splashsurf_b200 import io, __main__ as cli
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "import sys; sys.path.insert(0, %r); import oracle; oracle.reference().run_splashsurf(['splashsurf'] + sys.argv[1:])" % root
    args = ["reconstruct", os.path.join(GOLDEN, "reference_data", "bunny_frame_14_7705_particles.vtk"), "-r=0.025", "-l=2.0", "-c=0.5",
            "-a", "velocity", "-a", "id", "--normals=on", "--mesh-smoothing-iters=2", "--mesh-smoothing-weights=on", "--output-smoothing-weights=on"]
    ref, ours = str(tmp_path / "ref.ply"), str(tmp_path / "ours.ply")

    def run_reference():
        subprocess.check_call([sys.executable, "-c", code, *args, "-o", ref, "-q"])
        v1, t1, _, a1 = io.read_ply_mesh(ref)
        rng = np.random.default_rng(0)
        sv = np.sort(rng.choice(len(v1), 3000, replace=False))
        st = np.sort(rng.choice(len(t1), 4000, replace=False))
        np.savez_compressed(os.path.join(GOLDEN, "bunny_cli_ref.npz"), vertices=v1[sv], triangle_corners=v1[t1[st].astype(np.int64)],
                            **{"attr_" + k: a1[k][sv] for k in a1})
        return {"file_size": os.path.getsize(ref), "attributes": list(a1), "nv": len(v1), "nt": len(t1)}
    want = reference_output("bunny_cli_end_to_end", run_reference)
    assert cli.main(args + ["-o", ours]) == 0
    assert os.path.getsize(ours) == want["file_size"]
    g = load_golden("bunny_cli_ref")
    v2, t2, _, a2 = io.read_ply_mesh(ours)
    assert list(a2) == want["attributes"] == ["wnn", "sw", "normals", "velocity", "id"] and len(v2) == want["nv"] > 40000 and len(t2) == want["nt"]
    tree = cKDTree(v2)
    d, idx = tree.query(g["vertices"])
    assert d.max() < 2e-6 and len(np.unique(idx)) == len(idx)
    for k in want["attributes"]:
        r = g["attr_" + k]
        assert np.abs(r - a2[k][idx]).max() <= 5e-6 * max(1.0, float(np.abs(r).max())) + 2e-5, k
    corners = g["triangle_corners"]
    d, cidx = tree.query(corners.reshape(-1, 3))
    assert d.max() < 2e-6
    mine = set(map(tuple, np.sort(t2.astype(np.int64), axis=1)))
    assert all(tuple(tri) in mine for tri in np.sort(cidx.reshape(-1, 3), axis=1))
    with pytest.raises(ValueError, match='Missing attribute\\(s\\) "pressure" in input file'):
        cli.main(args[:5] + ["-a", "pressure"])
