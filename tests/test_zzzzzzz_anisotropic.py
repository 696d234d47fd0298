"""Anisotropic-kernel reconstruction (Yu & Turk 2013; DESIGN.md "Anisotropic kernels") against a float64 numpy model of its
definition, plus its behaviour and interfaces.

GPU-marked tests also run on the CPU executor: SS_TEST_EMULATED=1 python -m pytest tests/test_zzzzzzz_anisotropic.py -m gpu
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.spatial import cKDTree

from test_zzzz_reference_datasets import _canonical_mesh

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "golden", "reference_data")
GOLDEN = os.path.join(ROOT, "tests", "golden", "aniso_executor.npz")
KW = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=0.5, iso_surface_threshold=0.6)
R = 4 * 0.025                   # compact support radius of KW
CS = 0.5 * 0.025                # cube size of KW
# f32-scaled tolerances of the product against the float64 model: the moments are f32 sums of ~30 terms and the covariance
# subtracts mu mu^T; M depends on C / sigma_1 with a condition number up to max_ratio^2 = 16
TOL_CENTER = 1e-5 * R           # absolute, on x_bar
TOL_M = 2e-3                    # relative to max |M| (>= 1) of the particle
TOL_F = 2e-3                    # relative
TOL_L = 2e-3                    # relative to the largest level-set value of the tile


# ---------------------------------------------------------------------------- float64 model ----
def model_particles(p, rho, *, max_ratio=4.0, min_neighbors=10, smoothing=0.9, r=0.025, rest_density=1000.0):
    """Steps 1-4 of the definition in float64: centres (n, 3), matrices (n, 6) xx xy xz yy yz zz, factors (n,)."""
    p = np.asarray(p, np.float64)
    m = float(np.float32(np.float32(2 * r) ** 3 * np.float32(rest_density)))
    tree = cKDTree(p)
    xbar, mats, facs = np.empty_like(p), np.empty((len(p), 6)), np.empty(len(p))
    for i, nb in enumerate(tree.query_ball_point(p, R)):
        d = p[[j for j in nb if j != i]] - p[i]
        d = d[np.einsum("ij,ij->i", d, d) < R * R]
        w = 1.0 - (np.linalg.norm(d, axis=1) / R) ** 3
        W = 1.0 + w.sum()
        mu = (w[:, None] * d).sum(0) / W
        cov = (w[:, None, None] * d[:, :, None] * d[:, None, :]).sum(0) / W - np.outer(mu, mu)
        xbar[i] = p[i] + smoothing * mu
        ev, Q = np.linalg.eigh(cov)
        f = m / float(rho[i])
        M = np.eye(3)
        if len(d) >= min_neighbors and ev[-1] > 0:
            t = np.maximum(ev, ev[-1] / max_ratio) / ev[-1]
            M = Q @ np.diag(1.0 / t ** 2) @ Q.T
            f /= np.prod(t)
        mats[i] = M[[0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]
        facs[i] = f
    return xbar, mats, facs


def w_spline(d):
    """The cubic spline of the isotropic level set, support R (kernel.rs:61-107)."""
    q = 2.0 * np.asarray(d) / R
    f = np.where(q < 1.0, 1.5 / np.pi * (2.0 / 3.0 - q * q + 0.5 * q ** 3), np.where(q < 2.0, 0.25 / np.pi * (2.0 - q) ** 3, 0.0))
    return 8.0 / R ** 3 * f


def model_levelset(points, xbar, mats, facs):
    """Step 5: L(x) = sum_i f_i W_R(sqrt(u^T M_i u)) at points (k, 3)."""
    Ms = np.empty((len(mats), 3, 3))
    for e, (a, b) in enumerate(zip([0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2])):
        Ms[:, a, b] = Ms[:, b, a] = mats[:, e]
    out = np.zeros(len(points))
    tree = cKDTree(xbar)
    for k, nb in enumerate(tree.query_ball_point(points, R)):
        if not nb:
            continue
        u = points[k] - xbar[nb]
        q2 = np.einsum("ni,nij,nj->n", u, Ms[nb], u)
        out[k] = (facs[nb] * np.where(q2 < R * R, w_spline(np.sqrt(np.maximum(q2, 0.0))), 0.0)).sum()
    return out


def grid_points(grid, shape, origin_idx=(0, 0, 0)):
    mn = np.asarray(grid.aabb.min, np.float64)
    idx = np.stack(np.meshgrid(*[np.arange(o, o + s) for o, s in zip(origin_idx, shape)], indexing="ij"), -1).reshape(-1, 3)
    return mn + idx * np.float64(np.float32(CS))


# ---------------------------------------------------------------------------- clouds ----
def jittered_block(n=9, seed=1):
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(n)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.05
    return (g + rng.uniform(-0.01, 0.01, g.shape)).astype(np.float32)


def block_and_droplets(seed=2):
    rng = np.random.default_rng(seed)
    drops = rng.uniform([-0.3, -0.3, 0.6], [0.7, 0.7, 0.9], (12, 3))
    return np.concatenate([jittered_block(8, seed), drops]).astype(np.float32)


def sheet(n=14, seed=3):
    """One layer of particles in the plane z = 0.2 (spacing 2 r, jittered in-plane only)."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 2) * 0.05
    g = g + rng.uniform(-0.008, 0.008, g.shape)
    return np.c_[g, np.full(len(g), 0.2)].astype(np.float32)


def cube_2366():
    from splashsurf_b200 import io
    return np.ascontiguousarray(io.read_particles(os.path.join(DATA, "cube_2366_particles.vtk")), dtype=np.float32)


CLOUDS = {"block": jittered_block, "droplets": block_and_droplets, "sheet": sheet, "cube_2366": cube_2366}


def _aniso(ss, p, ctx=None, **kw):
    return ss.reconstruct_surface(p, context=ctx, anisotropic=True, **{**KW, "subdomain_num_cubes_per_dim": 16, **kw})


def _canon_tris(t):
    t = np.asarray(t, np.int64)
    if not len(t):
        return t.reshape(0, 3)
    t = np.stack([np.roll(row, -s) for row, s in zip(t, np.argmin(t, axis=1))])
    return t[np.lexsort(t.T[::-1])]


def _mesh_close(a_v, a_t, b_v, b_t, vtol):
    """Same triangle set with every vertex of a within vtol of its (one-to-one) partner in b."""
    a_v, b_v = np.asarray(a_v, np.float64), np.asarray(b_v, np.float64)
    assert a_v.shape == b_v.shape and len(a_t) == len(b_t), (a_v.shape, b_v.shape, len(a_t), len(b_t))
    if not len(a_v):
        return
    d, j = cKDTree(b_v).query(a_v)
    assert d.max() <= vtol and len(np.unique(j)) == len(j), d.max()
    assert np.array_equal(_canon_tris(j[np.asarray(a_t, np.int64)]), _canon_tris(b_t))


# ---------------------------------------------------------------------------- 1. per-particle data ----
@pytest.mark.gpu
@pytest.mark.parametrize("cloud", list(CLOUDS))
def test_particle_data_matches_model(ss, cloud):
    p = CLOUDS[cloud]()
    g = _aniso(ss, p, with_debug=True)
    xbar, mats, facs = model_particles(p, g.particle_densities)
    assert np.abs(g.anisotropic_centers - xbar).max() <= TOL_CENTER
    scale = np.maximum(np.abs(mats).max(axis=1, keepdims=True), 1.0)
    assert (np.abs(g.anisotropic_matrices - mats) / scale).max() <= TOL_M
    assert (np.abs(g.anisotropic_factors - facs) / facs).max() <= TOL_F
    assert 1 <= g.timings["anisotropy_max_jacobi_sweeps"] <= 8


# ---------------------------------------------------------------------------- 2. level set ----
@pytest.mark.gpu
@pytest.mark.parametrize("subdomain_grid", [True, False])
def test_levelset_tile_matches_model(ss, subdomain_grid):
    p = block_and_droplets()
    S = 16 if subdomain_grid else 64
    g0 = _aniso(ss, p, with_debug=True, subdomain_grid=subdomain_grid, subdomain_num_cubes_per_dim=S)
    xbar, mats, facs = model_particles(p, g0.particle_densities)
    # the tile that holds the block's corner particle (on the surface)
    corner = xbar[np.argmin(xbar.sum(axis=1))]
    ijk = np.floor((corner - np.asarray(g0.grid.aabb.min, np.float64)) / (S * np.float64(np.float32(CS)))).astype(int)
    nsd = [(c + S - 1) // S for c in g0.grid.ncells_per_dim]
    flat = int((ijk[0] * nsd[1] + ijk[1]) * nsd[2] + ijk[2])
    g = _aniso(ss, p, keep_levelset_tile_of=flat, subdomain_grid=subdomain_grid, subdomain_num_cubes_per_dim=S)
    pts = grid_points(g.grid, (S + 1,) * 3, tuple(ijk * S))
    ref = model_levelset(pts, xbar, mats, facs).reshape((S + 1,) * 3)
    assert ref.max() > 0.6
    assert np.abs(g.levelset_tile - ref).max() <= TOL_L * ref.max()


# ---------------------------------------------------------------------------- 3. mesh ----
@pytest.mark.gpu
def test_mesh_matches_model_field(ss):
    # the first seed whose model field has no grid value within TOL_MESH of the threshold (where the product's rounding could put
    # a point on the other side)
    TOL_MESH = 1e-5
    for seed in range(40):
        p = jittered_block(4, seed=100 + seed)
        g = _aniso(ss, p, with_debug=True, subdomain_grid=False)
        xbar, mats, facs = model_particles(p, g.particle_densities)
        shape = tuple(g.grid.npoints_per_dim)
        field = model_levelset(grid_points(g.grid, shape), xbar, mats, facs)
        if np.abs(field - 0.6).min() > TOL_MESH * field.max():
            break
    assert np.abs(field - 0.6).min() > TOL_MESH * field.max(), "no seed without a model value within the tolerance of the threshold"
    mc = ss.marching_cubes(field.reshape(shape).astype(np.float32), iso_surface_threshold=0.6, cube_size=float(np.float32(CS)),
                           translation=np.asarray(g.grid.aabb.min, np.float32))
    _mesh_close(g.mesh.vertices, g.mesh.triangles, mc.vertices, mc.triangles, 1e-4 * CS)


# ---------------------------------------------------------------------------- 4. reduction to isotropic ----
@pytest.mark.gpu
@pytest.mark.parametrize("data", ["bunny_frame_14_7705_particles.vtk", "dam_break_frame_9_6859_particles.bgeo"])
def test_reduces_to_isotropic(ss, data):
    from splashsurf_b200 import io
    p = np.ascontiguousarray(io.read_particles(os.path.join(DATA, data)), dtype=np.float32)
    kw = dict(particle_radius=0.025, smoothing_length=2.0, cube_size=1.0, iso_surface_threshold=0.6, subdomain_num_cubes_per_dim=32)
    iso = ss.reconstruct_surface(p, **kw)
    an = ss.reconstruct_surface(p, anisotropic=True, anisotropy_max_ratio=1.0, anisotropy_smoothing=0.0, **kw)
    _mesh_close(an.mesh.vertices, an.mesh.triangles, iso.mesh.vertices, iso.mesh.triangles, 1e-3 * 0.025)


@pytest.mark.gpu
def test_isolated_particle_is_isotropic(ss):
    p = np.array([[0.1, 0.2, 0.3]], np.float32)
    iso = ss.reconstruct_surface(p, **KW)
    for kw in (dict(), dict(anisotropy_max_ratio=8.0, anisotropy_min_neighbors=0, anisotropy_smoothing=1.0)):
        an = _aniso(ss, p, with_debug=True, **kw)
        assert np.array_equal(an.anisotropic_matrices, [[1, 0, 0, 1, 0, 1]]) and np.array_equal(an.anisotropic_centers, p)
        _mesh_close(an.mesh.vertices, an.mesh.triangles, iso.mesh.vertices, iso.mesh.triangles, 1e-6)


# ---------------------------------------------------------------------------- 5. behaviour ----
@pytest.mark.gpu
def test_sheet_is_thinner(ss):
    p = sheet()
    iso = ss.reconstruct_surface(p, **KW, subdomain_num_cubes_per_dim=16)
    an = _aniso(ss, p)
    assert iso.mesh.nvertices and an.mesh.nvertices
    # away from the rim, whose particles have fewer than min_neighbors neighbours and keep isotropic kernels
    inner = lambda v: v[((v[:, :2] > 0.15) & (v[:, :2] < 0.5)).all(axis=1)]                  # noqa: E731
    thick = lambda v: np.abs(inner(v)[:, 2].astype(np.float64) - 0.2).max()                 # noqa: E731
    assert thick(an.mesh.vertices) < thick(iso.mesh.vertices)


@pytest.mark.gpu
def test_translation_by_whole_cubes(ss):
    p = block_and_droplets()
    a = _aniso(ss, p)
    shift = np.float32(CS) * np.array([16, 32, 48], np.float32) * 4       # whole subdomains as well: the same decomposition
    b = _aniso(ss, p + shift)
    _mesh_close(b.mesh.vertices - shift, b.mesh.triangles, a.mesh.vertices, a.mesh.triangles, 4e-3 * CS)


@pytest.mark.gpu
def test_subdomain_and_global_paths_agree(ss):
    p = block_and_droplets()
    a = _aniso(ss, p)
    b = _aniso(ss, p, subdomain_grid=False)
    _mesh_close(a.mesh.vertices, a.mesh.triangles, b.mesh.vertices, b.mesh.triangles, 1e-5)


# ---------------------------------------------------------------------------- 6. determinism, pooled scratch ----
def _raw(r):
    return r.mesh.vertices.copy(), r.mesh.triangles.copy()


@pytest.mark.gpu
def test_bitwise_determinism_and_context_history(ss):
    p = block_and_droplets()
    fresh = {}
    for mode in (False, True):
        ctx = ss.Context(0)
        fresh[mode] = _raw(ss.reconstruct_surface(p, context=ctx, anisotropic=mode, **KW, subdomain_num_cubes_per_dim=16))
        again = _raw(ss.reconstruct_surface(p, context=ctx, anisotropic=mode, **KW, subdomain_num_cubes_per_dim=16))
        assert all(np.array_equal(x, y) for x, y in zip(fresh[mode], again))
        ctx.close()
    ctx = ss.Context(0)
    for mode in (False, True, False, True):
        got = _raw(ss.reconstruct_surface(p, context=ctx, anisotropic=mode, **KW, subdomain_num_cubes_per_dim=16))
        assert all(np.array_equal(x, y) for x, y in zip(fresh[mode], got)), mode
    ctx.close()


@pytest.mark.gpu
def test_matches_executor_fixture_bit_for_bit(ss):
    """The fixture was recorded on the CPU executor (tests/emul/cuda_emul.h); the B200 must compute the same bits."""
    g = _aniso(ss, jittered_block(6, seed=5), with_debug=True)
    ref = np.load(GOLDEN)
    for k in ("vertices", "triangles"):
        assert np.array_equal(getattr(g.mesh, k), ref[k]), k
    for k in ("centers", "matrices", "factors"):
        assert np.array_equal(getattr(g, "anisotropic_" + k), ref[k]), k


# ---------------------------------------------------------------------------- 7. interfaces ----
@pytest.mark.gpu
def test_invalid_parameters_raise(ss):
    p = jittered_block(4)
    for bad in (dict(anisotropy_max_ratio=0.5), dict(anisotropy_max_ratio=float("nan")), dict(anisotropy_smoothing=1.5),
                dict(anisotropy_smoothing=-0.1), dict(anisotropy_smoothing=float("nan"))):
        with pytest.raises(ss.SplashsurfError):
            _aniso(ss, p, **bad)
    with pytest.raises(ValueError):
        _aniso(ss, p, anisotropy_min_neighbors=-1)
    with pytest.raises(ValueError):
        _aniso(ss, p, sph_normals=True)
    with pytest.raises(ValueError):
        ss.reconstruction_pipeline(p, anisotropic=True, compute_normals=True, sph_normals=True, **KW)
    assert ss.reconstruct_surface(p, **KW).mesh.nvertices          # the context is usable afterwards


@pytest.mark.gpu
def test_partitioned_entry_refuses_anisotropy(ss):
    L = ss.load_library() if ss._LIB is None else ss._LIB
    ctx = ss.Context(0)
    a = ss._Anisotropy(4.0, 10, 0.9)
    assert L.ss_context_set_anisotropy_f32(ctx._h, C.byref(a)) == 0
    p = jittered_block(4)
    prm = ss.make_params(**KW, subdomain_num_cubes_per_dim=16)
    grid = ss._Grid()
    assert L.ss_grid_for_reconstruction_f32(ctx._h, p.ctypes.data, len(p), C.byref(prm), C.byref(grid)) == 0
    out = C.c_void_p()
    rc = L.ss_reconstruct_partition_f32(ctx._h, p.ctypes.data, len(p), C.byref(prm), C.byref(grid), 0, 0, 1, 0, 0, 0, C.byref(out))
    assert rc == 7 and b"anisotropic" in L.ss_last_error()
    ctx.close()


def test_distributed_and_cli_partition_refuse_anisotropy():
    from splashsurf_b200.distributed import DistributedReconstructor
    with pytest.raises(ValueError, match="anisotropic"):
        DistributedReconstructor(anisotropic=True, particle_radius=0.025, smoothing_length=2.0, cube_size=0.5)
    r = subprocess.run([sys.executable, "-m", "splashsurf_b200", "reconstruct", "in.vtk", "-r", "0.025", "-l", "2", "-c", "0.5",
                        "--partition=on", "--anisotropic=on"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode != 0 and "--anisotropic=on" in r.stderr


@pytest.mark.gpu
def test_pipeline_runs_on_anisotropic_mesh(ss):
    p = block_and_droplets()
    vel = np.random.default_rng(0).standard_normal((len(p), 3)).astype(np.float32)
    out, rec = ss.reconstruction_pipeline(p, anisotropic=True, mesh_smoothing_iters=3, compute_normals=True, attributes_to_interpolate={"v": vel},
                                          with_debug=True, **KW, subdomain_num_cubes_per_dim=16)
    assert out.nvertices == rec.mesh.nvertices > 0 and rec.anisotropic_factors is not None
    assert out.point_attributes["normals"].shape == (out.nvertices, 3) and out.point_attributes["v"].shape == (out.nvertices, 3)
    assert np.isfinite(out.point_attributes["v"]).all()


@pytest.mark.gpu
def test_cli_writes_the_python_mesh(ss, tmp_path):
    from splashsurf_b200 import __main__ as cli
    p = block_and_droplets()
    src = tmp_path / "in.xyz"
    p.tofile(src)
    dst = tmp_path / "out.ply"
    assert cli.main(["reconstruct", str(src), "-r", "0.025", "-l", "2", "-c", "0.5", "--subdomain-cubes", "16", "--anisotropic=on",
                     "-o", str(dst), "-q"]) in (0, None)
    ref = tmp_path / "ref.ply"
    g = _aniso(ss, p)
    ss.write_mesh(ref, g.mesh)
    assert dst.read_bytes() == ref.read_bytes()
