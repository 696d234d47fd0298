"""splashsurf_b200 -- B200-native surface reconstruction behind the splashsurf API.

Host-side mirror of the reference's Python front-end for the hot path
(``pysplashsurf.reconstruct_surface``, pysplashsurf/src/reconstruction.rs:128-207): same keyword names,
same RELATIVE ``smoothing_length`` / ``cube_size`` convention (both are multiplied by ``particle_radius``,
reconstruction.rs:172-176), same result attributes (``mesh.vertices`` (V,3) float32, ``mesh.triangles``
(T,3) uint64, ``particle_densities``, ``grid``, ``subdomain_grid``, ``particle_inside_aabb``).

The module mirrors every public name of ``pysplashsurf`` (``import splashsurf_b200 as pysplashsurf``; INTEGRATION.md lists what differs).

All compute happens in ``libsplashsurf_b200.so`` (hand-written sm_100a CUDA behind the C ABI declared in
``include/splashsurf_b200.h``).  There is no CPU fallback: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from enum import Enum
from typing import Optional, Sequence

import numpy as np

from . import build as _build

# every public name of the reference's Python module (tests/test_abi.py) + the extras of this package
__all__ = ["reconstruct_surface", "reconstruction_pipeline", "marching_cubes", "marching_cubes_cleanup", "barnacle_decimation", "convert_tris_to_quads",
           "laplacian_smoothing_parallel", "laplacian_smoothing_normals_parallel", "check_mesh_consistency", "neighborhood_search_spatial_hashing_parallel",
           "SphInterpolator", "run_splashsurf", "run_pysplashsurf", "TriMesh3d", "MixedTriQuadMesh3d", "MeshWithData", "MeshAttribute", "MeshType",
           "SurfaceReconstruction", "UniformGrid", "Aabb3d", "NeighborhoodLists", "VertexVertexConnectivity",
           "density_grid_loop", "write_mesh", "Context", "default_context", "make_params", "SplashsurfError", "library_path", "load_library"]

_HERE = os.path.dirname(os.path.abspath(__file__))


class SplashsurfError(RuntimeError):
    """Raised for every non-zero return of the C ABI (code + the library's message)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[ss error {code}] {message}")
        self.code = code
        self.message = message


# error codes of the C ABI (include/splashsurf_b200.h)
SS_OK, SS_ERR_INVALID_CELL_SIZE, SS_ERR_DEGENERATE_AABB, SS_ERR_INCONSISTENT_AABB, SS_ERR_INDEX_TOO_SMALL, SS_ERR_REAL_TOO_SMALL = 0, 1, 2, 3, 4, 5
SS_ERR_INVALID_PARAMETER, SS_ERR_UNSUPPORTED, SS_ERR_INVALID_DOMAIN = 6, 7, 8
SS_ERR_CUDA, SS_ERR_NO_DEVICE, SS_ERR_OUT_OF_MEMORY, SS_ERR_IO = 100, 101, 102, 103
SS_ERR_MESH_CHECK = 200      # Python mirror only: a mesh consistency check of reconstruction_pipeline failed (the reference returns an error)


class _Params(C.Structure):
    _fields_ = [
        ("particle_radius", C.c_float), ("rest_density", C.c_float), ("compact_support_radius", C.c_float),
        ("cube_size", C.c_float), ("iso_surface_threshold", C.c_float),
        ("has_particle_aabb", C.c_int32), ("particle_aabb_min", C.c_float * 3), ("particle_aabb_max", C.c_float * 3),
        ("enable_multi_threading", C.c_int32), ("enable_simd", C.c_int32), ("spatial_decomposition", C.c_int32),
        ("subdomain_num_cubes_per_dim", C.c_uint32), ("auto_disable", C.c_int32), ("global_neighborhood_list", C.c_int32),
    ]


class _Grid(C.Structure):
    _fields_ = [("aabb_min", C.c_float * 3), ("aabb_max", C.c_float * 3), ("cell_size", C.c_float),
                ("points_per_dim", C.c_int64 * 3), ("cells_per_dim", C.c_int64 * 3)]


class _Timings(C.Structure):
    _fields_ = [("upload", C.c_float), ("aabb_and_grid", C.c_float), ("decomposition", C.c_float), ("density", C.c_float),
                ("binning", C.c_float), ("levelset", C.c_float), ("marching_cubes", C.c_float), ("stitching", C.c_float),
                ("total_device", C.c_float), ("kernel_launches", C.c_uint64), ("levelset_launches", C.c_uint64),
                ("levelset_fixup_points", C.c_uint64), ("levelset_pairs", C.c_double),
                ("bricks_total", C.c_uint64), ("bricks_levelset", C.c_uint64), ("bricks_mc", C.c_uint64), ("bricks_fixscan", C.c_uint64),
                ("levelset_cert_evals", C.c_double), ("tile_setup", C.c_double)]


class _Anisotropy(C.Structure):
    """ss_anisotropy_f32 (include/splashsurf_b200.h)."""
    _fields_ = [("max_ratio", C.c_float), ("min_neighbors", C.c_uint32), ("smoothing", C.c_float)]


_LIB = None


def library_path() -> str:
    return _build.LIB


def load_library():
    """dlopen the in-tree CUDA library; raises if it has not been built (`python -m splashsurf_b200.build`)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: the CUDA extension has not been built "
                          f"(run `python -m splashsurf_b200.build`); there is no CPU fallback")
    _LIB = _bind(C.CDLL(path))
    return _LIB


class _MeshAttribute(C.Structure):
    """ss_mesh_attribute (include/splashsurf_b200.h)."""
    _fields_ = [("name", C.c_char_p), ("kind", C.c_int32), ("data", C.c_void_p)]


def _bind(L):
    """Declares the C-ABI prototypes (include/splashsurf_b200.h) on a loaded library handle."""
    vp, u64, i64 = C.c_void_p, C.c_uint64, C.c_int64
    L.ss_abi_version.restype = C.c_int
    L.ss_last_error.restype = C.c_char_p
    L.ss_context_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.ss_context_destroy.argtypes = [vp]
    L.ss_context_destroy.restype = None
    L.ss_reconstruct_surface_f32.argtypes = [vp, vp, u64, C.POINTER(_Params), C.POINTER(vp)]
    L.ss_surface_free.argtypes = [vp]
    L.ss_surface_free.restype = None
    L.ss_grid_for_reconstruction_f32.argtypes = [vp, vp, u64, C.POINTER(_Params), C.POINTER(_Grid)]
    for name in ("ss_surface_num_vertices", "ss_surface_num_triangles", "ss_surface_num_particles", "ss_surface_num_subdomains"):
        getattr(L, name).argtypes = [vp]
        getattr(L, name).restype = u64
    L.ss_surface_used_decomposition.argtypes = [vp]
    L.ss_surface_grid.argtypes = [vp, C.POINTER(_Grid)]
    L.ss_surface_subdomain_grid.argtypes = [vp, C.POINTER(_Grid)]
    for name in ("ss_surface_copy_vertices", "ss_surface_copy_triangles_u32", "ss_surface_copy_triangles_u64",
                 "ss_surface_copy_particle_densities", "ss_surface_copy_particle_inside_aabb",
                 "ss_surface_copy_vertex_edge_keys", "ss_surface_copy_levelset_tile"):
        getattr(L, name).argtypes = [vp, vp]
    for name in ("ss_surface_device_vertices", "ss_surface_device_triangles", "ss_surface_device_densities"):
        getattr(L, name).argtypes = [vp]
        getattr(L, name).restype = vp
    L.ss_surface_copy_subdomains.argtypes = [vp, vp, vp, vp]
    L.ss_surface_num_neighbors.argtypes = [vp]
    L.ss_surface_num_neighbors.restype = u64
    L.ss_surface_copy_neighbor_lists.argtypes = [vp, vp, vp]
    L.ss_context_keep_levelset_tile.argtypes = [vp, i64]
    L.ss_surface_timings.argtypes = [vp, C.POINTER(_Timings)]
    L.ss_context_set_tile_batch.argtypes = [vp, C.c_uint32]
    L.ss_context_set_levelset_exact_everywhere.argtypes = [vp, C.c_int]
    L.ss_context_set_levelset_variant.argtypes = [vp, C.c_int]
    L.ss_context_set_density_variant.argtypes = [vp, C.c_int]
    L.ss_context_set_mc_variant.argtypes = [vp, C.c_int]
    L.ss_context_set_copy_chunk_bytes.argtypes = [vp, u64]
    L.ss_context_set_count_pairs.argtypes = [vp, C.c_int]
    L.ss_context_set_compute_sph_normals.argtypes = [vp, C.c_int]
    L.ss_surface_copy_normals.argtypes = [vp, vp]
    L.ss_context_set_anisotropy_f32.argtypes = [vp, C.POINTER(_Anisotropy)]
    L.ss_surface_copy_anisotropy_f32.argtypes = [vp, vp, vp, vp]
    L.ss_surface_anisotropy_stats.argtypes = [vp, vp, vp]
    L.ss_surface_device_normals.argtypes = [vp]
    L.ss_surface_device_normals.restype = vp
    L.ss_levelset_tile_f32.argtypes = [vp, vp, vp, u64, vp, C.c_float, vp, C.c_uint32, C.c_float, C.c_float, C.c_int, vp]
    L.ss_reconstruct_partition_f32.argtypes = [vp, vp, u64, C.POINTER(_Params), C.POINTER(_Grid), C.c_int, i64, i64, i64, u64, C.c_int, C.POINTER(vp)]
    L.ss_reconstruct_partition_cb_f32.argtypes = [vp, vp, u64, C.POINTER(_Params), C.POINTER(_Grid), C.c_int, i64, i64, i64, vp, vp, C.POINTER(vp)]
    L.ss_partition_stats_f32.argtypes = [vp, vp, u64, C.POINTER(_Grid), C.c_uint32, C.c_int, vp, vp]
    L.ss_partition_members_f32.argtypes = [vp, vp, u64, C.POINTER(_Params), C.POINTER(_Grid), C.c_int, vp, vp]
    L.ss_partition_pack_f32.argtypes = [vp, vp, u64, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_uint64), vp]
    L.ss_surface_max_subdomain_particles.argtypes = [vp]
    L.ss_surface_max_subdomain_particles.restype = u64
    L.ss_surface_device_vertex_keys.argtypes = [vp]
    L.ss_surface_device_vertex_keys.restype = vp
    L.ss_surface_copy_subdomain_owned.argtypes = [vp, vp]
    L.ss_weld_meshes.argtypes = [vp, vp, vp, u64, vp, u64, vp, u64, C.POINTER(u64)]
    L.ss_surface_interpolate_quantity_f32.argtypes = [vp, vp, C.c_uint32, C.c_int, vp]
    L.ss_surface_compute_smoothing_weights_f32.argtypes = [vp, C.c_float, vp, vp]
    L.ss_surface_laplacian_smoothing_f32.argtypes = [vp, C.c_uint32, C.c_float, vp]
    L.ss_marching_cubes_tiles_f32.argtypes = [vp, vp, C.c_uint32, vp, vp, C.c_float, C.c_float, C.POINTER(vp)]
    L.ss_neighborhood_search_f32.argtypes = [vp, vp, C.c_uint64, vp, vp, C.c_float, C.POINTER(vp)]
    L.ss_sph_interpolator_create_f32.argtypes = [vp, vp, C.c_uint64, vp, C.c_float, C.c_float, C.POINTER(vp)]
    L.ss_sph_interpolate_quantity_at_f32.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint64, C.c_int, vp]
    L.ss_sph_interpolate_normals_at_f32.argtypes = [vp, vp, C.c_uint64, vp]
    L.ss_surface_compute_normals_f32.argtypes = [vp, C.c_int]
    L.ss_surface_smooth_normals_f32.argtypes = [vp, C.c_uint32]
    L.ss_surface_vertex_connectivity.argtypes = [vp, vp, vp, C.POINTER(u64)]
    L.ss_surface_from_mesh_f32.argtypes = [vp, vp, u64, vp, u64, C.POINTER(vp)]
    L.ss_surface_set_normals_f32.argtypes = [vp, vp]
    L.ss_host_alloc_pinned.argtypes = [u64]
    L.ss_host_alloc_pinned.restype = vp
    L.ss_host_free_pinned.argtypes = [vp]
    L.ss_host_free_pinned.restype = None
    L.ss_surface_replace_mesh_f32.argtypes = [vp, vp, u64, vp, u64]
    L.ss_mesh_cleanup_f32.argtypes = [vp, C.POINTER(u64), vp, C.POINTER(u64), C.POINTER(_Grid), C.c_float, u64, C.c_int, vp, vp]
    L.ss_mesh_decimation_f32.argtypes = [vp, C.POINTER(u64), vp, C.POINTER(u64), C.c_int, vp, vp]
    L.ss_mesh_tris_to_quads_f32.argtypes = [vp, u64, vp, u64, C.c_float, C.c_float, C.c_float, vp, C.POINTER(u64), vp, C.POINTER(u64)]
    L.ss_write_mesh_f32.argtypes = [C.c_char_p, C.c_int, vp, u64, vp, u64, vp, u64, C.c_int, C.POINTER(_MeshAttribute), C.c_uint32,
                                    C.POINTER(_MeshAttribute), C.c_uint32, C.c_uint32]
    L.ss_format_f32.argtypes = [C.c_float, C.c_char_p, u64]
    L.ss_meshio_set_chunk_items.argtypes = [u64]
    if L.ss_abi_version() != 3:
        raise ImportError("libsplashsurf_b200.so ABI version mismatch")
    return L


def _check(L, rc: int):
    if rc != 0:
        raise SplashsurfError(rc, (L.ss_last_error() or b"").decode("utf-8", "replace"))


# ---------------------------------------------------------------------------- result types ----
@dataclass
class Aabb3d:
    """Mirrors pysplashsurf.Aabb3d (min / max corners; aabb.rs)."""
    min: np.ndarray
    max: np.ndarray

    @staticmethod
    def from_min_max(min, max) -> "Aabb3d":                # noqa: A002 - the reference's argument names
        return Aabb3d(np.asarray(min, dtype=np.float64).reshape(3).copy(), np.asarray(max, dtype=np.float64).reshape(3).copy())

    @staticmethod
    def from_points(points) -> "Aabb3d":
        """Smallest AABB around the points (aabb.rs `from_points`); zero-sized at the origin for an empty set."""
        pts = np.asarray(points).reshape(-1, 3)
        if len(pts) == 0:
            return Aabb3d(np.zeros(3), np.zeros(3))
        return Aabb3d(pts.min(axis=0).astype(np.float64), pts.max(axis=0).astype(np.float64))

    def contains_point(self, point) -> bool:
        """Half-open towards the max corner, like the reference."""
        q = np.asarray(point, dtype=np.float64).reshape(3)
        return bool(np.all(q >= np.asarray(self.min, np.float64)) and np.all(q < np.asarray(self.max, np.float64)))


@dataclass
class UniformGrid:
    """Mirrors pysplashsurf.UniformGrid / UniformCartesianCubeGrid3d (uniform_grid.rs:132-142)."""
    aabb: Aabb3d
    cell_size: float
    npoints_per_dim: list
    ncells_per_dim: list

    @staticmethod
    def _from(g: _Grid) -> "UniformGrid":
        return UniformGrid(Aabb3d(np.array(g.aabb_min, dtype=np.float32), np.array(g.aabb_max, dtype=np.float32)),
                           float(g.cell_size), [int(v) for v in g.points_per_dim], [int(v) for v in g.cells_per_dim])


@dataclass
class TriMesh3d:
    """Mirrors splashsurf_lib::mesh::TriMesh3d (mesh.rs:186-193)."""
    vertices: np.ndarray   # (V, 3) float32
    triangles: np.ndarray  # (T, 3) uint64 (usize in the reference)

    @property
    def nvertices(self) -> int:
        return len(self.vertices)

    @property
    def ncells(self) -> int:
        return len(self.triangles)

    @property
    def dtype(self):
        return np.dtype(np.float32)

    def copy(self) -> "TriMesh3d":
        return TriMesh3d(self.vertices.copy(), self.triangles.copy())

    def write_to_file(self, path, *, file_format: Optional[str] = None) -> None:
        """``pysplashsurf.TriMesh3d.write_to_file``; the file is the reference CLI's (`write_mesh`), by extension or `file_format`."""
        write_mesh(path, self, file_format=file_format)

    def vertex_normals_parallel(self, context=None) -> np.ndarray:
        """Area-weighted vertex normals on the device (TriMesh3d::par_vertex_normals, mesh.rs:799-906)."""
        with _MeshSurface(self.vertices, self.triangles, context) as m:
            _check(m.L, m.L.ss_surface_compute_normals_f32(m.s, 0))
            out = np.empty((self.nvertices, 3), np.float32)
            if len(out):
                _check(m.L, m.L.ss_surface_copy_normals(m.s, out.ctypes.data))
            return out

    def vertex_vertex_connectivity(self, context=None) -> "VertexVertexConnectivity":
        """Vertex-vertex connectivity computed on the device (mesh.rs:290-306; neighbours in ascending order)."""
        with _MeshSurface(self.vertices, self.triangles, context) as m:
            n = C.c_uint64()
            off = np.empty(self.nvertices + 1, np.uint64)
            _check(m.L, m.L.ss_surface_vertex_connectivity(m.s, off.ctypes.data, None, C.byref(n)))
            idx = np.empty(n.value, np.uint32)
            _check(m.L, m.L.ss_surface_vertex_connectivity(m.s, off.ctypes.data, idx.ctypes.data if len(idx) else None, C.byref(n)))
        return VertexVertexConnectivity(off, idx, np.asarray(self.triangles), self.nvertices)


class VertexVertexConnectivity:
    """Mirrors pysplashsurf.VertexVertexConnectivity (CSR storage; the triangles are kept so that device functions taking only
    a connectivity can rebuild it there)."""

    def __init__(self, offsets: np.ndarray, indices: np.ndarray, triangles: np.ndarray, nvertices: int):
        self.offsets, self.indices, self._triangles, self._nv = offsets, indices, triangles, int(nvertices)

    def copy_connectivity(self) -> list:
        return [self.indices[int(self.offsets[i]):int(self.offsets[i + 1])].tolist() for i in range(self._nv)]

    take_connectivity = copy_connectivity


def _grid_struct(grid: "UniformGrid") -> _Grid:
    g = _Grid()
    for d in range(3):
        g.aabb_min[d] = float(grid.aabb.min[d]); g.aabb_max[d] = float(grid.aabb.max[d])
        g.points_per_dim[d] = int(grid.npoints_per_dim[d]); g.cells_per_dim[d] = int(grid.ncells_per_dim[d])
    g.cell_size = float(grid.cell_size)
    return g


def _host_mesh_op(mesh: "TriMesh3d", call) -> "VertexVertexConnectivity":
    """Runs an in-place host mesh operation of the library (ss_mesh_*_f32) on `mesh` and returns the connectivity it reports."""
    L = load_library()
    v = np.ascontiguousarray(mesh.vertices, dtype=np.float32).copy()
    t = np.ascontiguousarray(mesh.triangles, dtype=np.uint32).copy()
    nv, nt = C.c_uint64(len(v)), C.c_uint64(len(t))
    off = np.zeros(len(v) + 1, np.uint64)
    idx = np.empty(max(6 * len(t), 1), np.uint32)           # sum of the valences = 2 x edges <= 6 x triangles (3 x for a closed mesh)
    _check(L, call(L, v.ctypes.data if len(v) else None, C.byref(nv), t.ctypes.data if len(t) else None, C.byref(nt), off.ctypes.data, idx.ctypes.data))
    mesh.vertices = v[:nv.value].copy()
    mesh.triangles = t[:nt.value].astype(np.uint64)
    off = off[:nv.value + 1].copy()
    return VertexVertexConnectivity(off, idx[:int(off[-1])].copy(), mesh.triangles, nv.value)


def marching_cubes_cleanup(mesh: "TriMesh3d", grid: "UniformGrid", *, max_rel_snap_dist: Optional[float] = None, max_iter: int = 5,
                           keep_vertices: bool = False) -> "VertexVertexConnectivity":
    """``pysplashsurf.marching_cubes_cleanup`` (postprocessing.rs:99-242): simplifies a marching-cubes mesh in place by merging
    vertices that share their nearest grid point; returns the vertex-vertex connectivity of the result.  Host code in the library
    (sequential half-edge collapses, as in the reference).  Accepts a TriMesh3d or a MeshWithData (its attributes are NOT carried over
    to the new vertex set; the pipeline applies the clean-up before any attribute exists)."""
    mesh = getattr(mesh, "mesh", mesh)
    g = _grid_struct(grid)
    snap = -1.0 if max_rel_snap_dist is None else float(max_rel_snap_dist)
    return _host_mesh_op(mesh, lambda L, v, nv, t, nt, off, idx: L.ss_mesh_cleanup_f32(v, nv, t, nt, C.byref(g), C.c_float(snap), int(max_iter),
                                                                                        int(bool(keep_vertices)), off, idx))


def barnacle_decimation(mesh: "TriMesh3d", *, keep_vertices: bool = False) -> "VertexVertexConnectivity":
    """``pysplashsurf.barnacle_decimation`` (postprocessing.rs:244-686): merges the single and double barnacle configurations of a
    marching-cubes mesh in place; returns the vertex-vertex connectivity of the result."""
    return _host_mesh_op(mesh, lambda L, v, nv, t, nt, off, idx: L.ss_mesh_decimation_f32(v, nv, t, nt, int(bool(keep_vertices)), off, idx))


@dataclass
class MixedTriQuadMesh3d:
    """Mirrors pysplashsurf.MixedTriQuadMesh3d (mesh.rs): vertices plus triangle and quad cells."""
    vertices: np.ndarray
    _triangles: np.ndarray
    _quads: np.ndarray

    def get_triangles(self) -> np.ndarray:
        return self._triangles

    def get_quads(self) -> np.ndarray:
        return self._quads

    @property
    def dtype(self):
        return np.dtype(np.float32)

    def copy(self) -> "MixedTriQuadMesh3d":
        return MixedTriQuadMesh3d(self.vertices.copy(), self._triangles.copy(), self._quads.copy())

    def write_to_file(self, path, *, file_format: Optional[str] = None) -> None:
        write_mesh(path, self, file_format=file_format)

    @property
    def nvertices(self) -> int:
        return len(self.vertices)

    @property
    def ncells(self) -> int:
        return len(self._triangles) + len(self._quads)


def convert_tris_to_quads(mesh: "TriMesh3d", *, non_squareness_limit: float = 1.75, normal_angle_limit: float = 10.0,
                          max_interior_angle: float = 135.0) -> MixedTriQuadMesh3d:
    """``pysplashsurf.convert_tris_to_quads`` (postprocessing.rs:689-910; angles in degrees): merges pairs of triangles sharing an edge
    into quads.  Returns a new mesh; the input is not modified.  Host code in the library, cells in the reference's order.  A
    MeshWithData comes back as a MeshWithData around the quad mesh with its point attributes (cell attributes are dropped, as in
    reconstruct.rs:1424-1437)."""
    if hasattr(mesh, "point_attributes"):
        q = convert_tris_to_quads(mesh.mesh, non_squareness_limit=non_squareness_limit, normal_angle_limit=normal_angle_limit, max_interior_angle=max_interior_angle)
        return MeshWithData(q, dict(mesh.point_attributes), {})
    L = load_library()
    v = np.ascontiguousarray(mesh.vertices, dtype=np.float32)
    t = np.ascontiguousarray(mesh.triangles, dtype=np.uint32)
    to = np.empty((max(len(t), 1), 3), np.uint32)
    qo = np.empty((max(len(t) // 2, 1), 4), np.uint32)
    nt, nq = C.c_uint64(0), C.c_uint64(0)
    rad = lambda deg: float(np.float32(float(deg) * (np.pi / 180.0)))      # f64::to_radians, then `as f32` (pysplashsurf/src/postprocessing.rs:45-58)
    _check(L, L.ss_mesh_tris_to_quads_f32(v.ctypes.data if len(v) else None, len(v), t.ctypes.data if len(t) else None, len(t),
                                          C.c_float(float(np.float32(non_squareness_limit))), C.c_float(rad(normal_angle_limit)),
                                          C.c_float(rad(max_interior_angle)), to.ctypes.data, C.byref(nt), qo.ctypes.data, C.byref(nq)))
    return MixedTriQuadMesh3d(v.copy(), to[:nt.value].astype(np.uint64), qo[:nq.value].astype(np.uint64))


def _edge_table(tris: np.ndarray):
    """Undirected edges of a triangle array: (unique sorted vertex pairs, incident face count per unique edge, inverse index per half-edge
    in (triangle, local edge) order)."""
    t = np.asarray(tris, dtype=np.int64)
    he = np.stack([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]], axis=1).reshape(-1, 2)      # half-edge (t, e) at row 3 t + e
    und = np.sort(he, axis=1)
    uniq, inv, cnt = np.unique(und, axis=0, return_inverse=True, return_counts=True)
    return uniq, cnt, inv.reshape(-1)


def find_non_manifold_vertices(mesh: "TriMesh3d") -> np.ndarray:
    """TriMesh3d::find_non_manifold_vertices (mesh.rs:1007-1090): vertices whose incident triangles do not form ONE fan, i.e. are not
    all connected through edges at that vertex.  Host code (numpy + scipy's connected components), ascending vertex index."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    t = np.asarray(mesh.triangles, dtype=np.int64)
    nt = len(t)
    if nt == 0:
        return np.zeros(0, np.int64)
    _, _, inv = _edge_table(t)
    # corner node id = 3 * triangle + local corner; half-edge (t, e) joins corners e and (e + 1) % 3 of triangle t to the same edge
    order = np.argsort(inv, kind="stable")
    same = inv[order][1:] == inv[order][:-1]
    a, b = order[:-1][same], order[1:][same]                   # consecutive half-edges of one undirected edge
    ta, ea, tb, eb = a // 3, a % 3, b // 3, b % 3
    va0, va1 = t[ta, ea], t[ta, (ea + 1) % 3]
    vb0 = t[tb, eb]
    # connect the corners that sit on the same vertex
    ca0, ca1 = 3 * ta + ea, 3 * ta + (ea + 1) % 3
    cb0, cb1 = 3 * tb + eb, 3 * tb + (eb + 1) % 3
    flip = vb0 != va0                                          # opposite orientation: b's first corner is a's second vertex
    src = np.concatenate([ca0, ca1])
    dst = np.concatenate([np.where(flip, cb1, cb0), np.where(flip, cb0, cb1)])
    n_nodes = 3 * nt
    g = coo_matrix((np.ones(len(src), np.int8), (src, dst)), shape=(n_nodes, n_nodes))
    _, label = connected_components(g, directed=False)
    vert_of_corner = t.reshape(-1)
    pairs = np.unique(np.stack([vert_of_corner, label], axis=1), axis=0)
    verts, fans = np.unique(pairs[:, 0], return_counts=True)
    return verts[fans > 1]


def check_mesh_consistency(mesh: "TriMesh3d", grid: "UniformGrid", *, check_closed: bool = True, check_manifold: bool = True,
                           debug: bool = False) -> Optional[str]:
    """``pysplashsurf.check_mesh_consistency`` (marching_cubes.rs:129-213): None if the mesh is closed (no edge with a single incident
    triangle) / manifold (no edge with more than two incident triangles, no vertex with more than one triangle fan), else a text with
    the reference's messages.  Host code.  Accepts a TriMesh3d or a MeshWithData."""
    mesh = getattr(mesh, "mesh", mesh)
    uniq, cnt, _ = _edge_table(mesh.triangles)
    n_boundary, n_nm_edges = int((cnt == 1).sum()), int((cnt > 2).sum())
    nm_verts = find_non_manifold_vertices(mesh)
    if (not check_closed or n_boundary == 0) and (not check_manifold or (n_nm_edges == 0 and len(nm_verts) == 0)):
        return None
    msgs = []
    if check_closed and n_boundary:
        msgs.append(f"Mesh is not closed. It has {n_boundary} boundary edges (edges that are connected to only one triangle).")
        if debug:
            msgs += [f"\tboundary edge {e.tolist()}" for e in uniq[cnt == 1]]
    if check_manifold and n_nm_edges:
        msgs.append(f"Mesh is not manifold. It has {n_nm_edges} non-manifold edges (edges that are connected to more than two triangles).")
        if debug:
            msgs += [f"\tnon-manifold edge {e.tolist()}" for e in uniq[cnt > 2]]
    if check_manifold and len(nm_verts):
        msgs.append(f"Mesh is not manifold. It has {len(nm_verts)} non-manifold vertices (vertices with more than one triangle fan).")
        if debug:
            msgs.append(f"\tNon-manifold vertices: {nm_verts.tolist()}")
    return "\n".join(msgs)


def find_flipped_faces(mesh: "TriMesh3d") -> np.ndarray:
    """The orientation check of the pipeline (reconstruct.rs:1481-1507): triangles whose unit normal makes an angle of more than 0.99 pi
    with the area-weighted normal of one of their vertices.  Host code; ascending triangle index."""
    v = np.asarray(mesh.vertices, dtype=np.float32)
    t = np.asarray(mesh.triangles, dtype=np.int64)
    if len(t) == 0:
        return np.zeros(0, np.int64)
    cr = np.cross(v[t[:, 1]] - v[t[:, 0]], v[t[:, 2]] - v[t[:, 0]]).astype(np.float32)        # area-weighted (mesh.rs:842-906)
    vn = np.zeros_like(v)
    for c in range(3):
        np.add.at(vn, t[:, c], cr)
    with np.errstate(invalid="ignore", divide="ignore"):
        tn = cr / np.linalg.norm(cr, axis=1, keepdims=True)
        n1 = vn[t]                                                                             # (T, 3 corners, 3)
        cang = np.einsum("tcd,td->tc", n1, tn) / (np.linalg.norm(n1, axis=2) * np.linalg.norm(tn, axis=1, keepdims=True))
        ang = np.arccos(np.clip(cang, -1.0, 1.0))
    return np.nonzero((ang > np.pi * 0.99).any(axis=1))[0]


def clamp_mesh_with_aabb(mesh: "TriMesh3d", aabb_min, aabb_max, *, clamp_vertices: bool = True, keep_vertices: bool = False, point_attributes=None):
    """Mesh3d::par_clamp_with_aabb (mesh.rs:334-371) as the pipeline applies it (reconstruct.rs:1394-1408): keeps the triangles with at
    least one vertex inside the half-open box [min, max) (aabb.rs:220-222), drops the vertices no kept triangle uses (unless
    `keep_vertices`), then clamps the remaining vertices into the box.  Returns (TriMesh3d, filtered point attributes).  Host code."""
    v = np.asarray(mesh.vertices, dtype=np.float32)
    t = np.asarray(mesh.triangles)
    mn, mx = np.asarray(aabb_min, np.float32), np.asarray(aabb_max, np.float32)
    inside = np.all(v >= mn, axis=1) & np.all(v < mx, axis=1)
    keep_t = inside[t.astype(np.int64)].any(axis=1) if len(t) else np.zeros(0, bool)
    t2 = t[keep_t]
    attrs = dict(point_attributes or {})
    if not keep_vertices:
        used = np.zeros(len(v), bool)
        used[t2.astype(np.int64).reshape(-1)] = True
        newid = np.cumsum(used) - 1
        v = v[used]
        t2 = newid[t2.astype(np.int64)].astype(t.dtype)
        attrs = {k: np.asarray(a)[used] for k, a in attrs.items()}
    v = np.clip(v, mn, mx) if clamp_vertices else v.copy()
    return TriMesh3d(np.ascontiguousarray(v, dtype=np.float32), t2), attrs


class _MeshSurface:
    """A device surface around an arbitrary triangle mesh (ss_surface_from_mesh_f32) for the mesh-only post-processing entries."""

    def __init__(self, vertices, triangles, context=None):
        self.ctx = context or default_context()
        self.L = self.ctx._L
        v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(triangles).reshape(-1, 3)
        if len(t) and int(t.max()) >= len(v):
            raise ValueError("triangle index out of range")
        t = np.ascontiguousarray(t, dtype=np.uint32)
        self.s = C.c_void_p()
        _check(self.L, self.L.ss_surface_from_mesh_f32(self.ctx._h, v.ctypes.data if len(v) else None, len(v), t.ctypes.data if len(t) else None,
                                                       len(t), C.byref(self.s)))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.ctx.free_surface(self.s)
        return False


def laplacian_smoothing_parallel(mesh, vertex_connectivity=None, *, iterations: int, beta: float = 1.0, weights, context=None) -> None:
    """``pysplashsurf.laplacian_smoothing_parallel``: weighted Laplacian smoothing of ``mesh.vertices`` in place
    (postprocessing.rs:17-53) on the device.  ``vertex_connectivity`` is accepted for signature parity; the device rebuilds it."""
    m0 = mesh.mesh if isinstance(mesh, MeshWithData) else mesh
    w = np.ascontiguousarray(weights, dtype=np.float32)
    if len(w) != m0.nvertices:
        raise ValueError("one weight per vertex is required")
    with _MeshSurface(m0.vertices, m0.triangles, context) as m:
        _check(m.L, m.L.ss_surface_laplacian_smoothing_f32(m.s, int(iterations), C.c_float(float(beta)), w.ctypes.data if len(w) else None))
        out = np.empty((m0.nvertices, 3), np.float32)
        _check(m.L, m.L.ss_surface_copy_vertices(m.s, out.ctypes.data if len(out) else None))
    m0.vertices[...] = out


def laplacian_smoothing_normals_parallel(normals: np.ndarray, vertex_connectivity: VertexVertexConnectivity, *, iterations: int, context=None) -> None:
    """``pysplashsurf.laplacian_smoothing_normals_parallel``: smooths the (N, 3) float32 normal field in place
    (postprocessing.rs:56-97) on the device."""
    n = np.asarray(normals)
    if n.dtype != np.float32 or n.ndim != 2 or n.shape[1] != 3 or len(n) != vertex_connectivity._nv:
        raise ValueError("normals must be a float32 array of shape (num_vertices, 3)")
    src = np.ascontiguousarray(n)
    with _MeshSurface(np.zeros((len(n), 3), np.float32), vertex_connectivity._triangles, context) as m:
        _check(m.L, m.L.ss_surface_set_normals_f32(m.s, src.ctypes.data if len(src) else None))
        _check(m.L, m.L.ss_surface_smooth_normals_f32(m.s, int(iterations)))
        out = np.empty_like(src)
        if len(out):
            _check(m.L, m.L.ss_surface_copy_normals(m.s, out.ctypes.data))
    normals[...] = out


class NeighborhoodLists:
    """Mirrors pysplashsurf.NeighborhoodLists on top of CSR arrays (offsets, indices)."""

    def __init__(self, offsets: np.ndarray, indices: np.ndarray):
        self.offsets, self.indices = offsets, indices

    def __len__(self) -> int:
        return len(self.offsets) - 1

    def __getitem__(self, idx: int) -> list:
        return self.indices[int(self.offsets[idx]):int(self.offsets[idx + 1])].tolist()

    def get_neighborhood_lists(self) -> list:
        return [self[i] for i in range(len(self))]


@dataclass
class SurfaceReconstruction:
    """Mirrors splashsurf_lib::SurfaceReconstruction<i64, f32> (lib.rs:247-262)."""
    mesh: TriMesh3d
    grid: UniformGrid
    subdomain_grid: Optional[UniformGrid]
    particle_densities: Optional[np.ndarray]
    particle_inside_aabb: Optional[np.ndarray]
    particle_neighbors: Optional[list] = None
    # extras of the device path
    timings: Optional[dict] = None
    vertex_edge_keys: Optional[np.ndarray] = None
    subdomains: Optional[dict] = None
    levelset_tile: Optional[np.ndarray] = None
    normals: Optional[np.ndarray] = None       # (V, 3) unit SPH normals when requested
    anisotropic_centers: Optional[np.ndarray] = None    # (N, 3) kernel centres x_bar (anisotropic, with_debug)
    anisotropic_matrices: Optional[np.ndarray] = None   # (N, 6) M = R^2 A: xx, xy, xz, yy, yz, zz
    anisotropic_factors: Optional[np.ndarray] = None    # (N,) f = (m / rho) R^3 / (a1 a2 a3)


# ---------------------------------------------------------------------------- context ----
class Context:
    """One GPU's stream + reusable device buffers (the analogue of the reference's rayon pool + workspace)."""

    def __init__(self, device: int = -1):
        self._L = load_library()
        h = C.c_void_p()
        _check(self._L, self._L.ss_context_create(int(device), C.byref(h)))
        self._h = h
        # opt-in: reconstruct_surface / reconstruction_pipeline return their big arrays (vertices, triangles, densities) as views of
        # page-locked buffers owned by this context -- no fresh pages, copies at PCIe speed -- that the NEXT reconstruction on the
        # context overwrites (copy what must outlive it)
        self.reuse_host_buffers = False

    def close(self):
        if getattr(self, "_h", None):
            self._free_host_pool()
            self._L.ss_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def host_array(self, name: str, shape, dtype) -> np.ndarray:
        """A numpy view of a page-locked host buffer owned by this context (grown on demand, reused by name): what
        `reuse_host_buffers` hands out as result arrays.  Valid until the next call that asks for the same name, or `close`."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        pool = self.__dict__.setdefault("_host_pool", {})
        ptr, cap = pool.get(name, (None, 0))
        if cap < n or ptr is None:
            if ptr:
                self._L.ss_host_free_pinned(ptr)
            cap = int(n * 1.25) + 4096
            ptr = self._L.ss_host_alloc_pinned(cap)
            if not ptr:
                pool.pop(name, None)
                raise MemoryError(f"cannot page-lock {cap} bytes for {name}")
            pool[name] = (ptr, cap)
        buf = (C.c_char * max(n, 1)).from_address(ptr)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def _free_host_pool(self):
        for ptr, _ in self.__dict__.get("_host_pool", {}).values():
            if ptr:
                self._L.ss_host_free_pinned(ptr)
        self.__dict__["_host_pool"] = {}

    def set_tile_batch(self, max_tiles: int):
        _check(self._L, self._L.ss_context_set_tile_batch(self._h, int(max_tiles)))

    def set_levelset_exact_everywhere(self, on: bool):
        """Evaluate every level-set grid point exactly (default: interior points are only classified)."""
        _check(self._L, self._L.ss_context_set_levelset_exact_everywhere(self._h, int(bool(on))))

    def set_levelset_variant(self, variant: int):
        """2 (default): warp-per-brick certification + exact kernels; 1: CTA-per-brick certification kernel; 0: fused kernel
        (same results)."""
        _check(self._L, self._L.ss_context_set_levelset_variant(self._h, int(variant)))

    def set_mc_variant(self, variant: int):
        """1 (default): warp-per-brick marching cubes + fix-up sweep; 0: CTA-per-brick passes (same mesh, other vertex order)."""
        _check(self._L, self._L.ss_context_set_mc_variant(self._h, int(variant)))

    def set_density_variant(self, variant: int):
        """0 (default): thread-per-particle kernel; 1 / 2: cell-cooperative kernel, candidates staged by bulk copies / by loads
        (same results; slower on the B200, kept as an experiment)."""
        _check(self._L, self._L.ss_context_set_density_variant(self._h, int(variant)))

    def set_count_pairs(self, on: bool):
        _check(self._L, self._L.ss_context_set_count_pairs(self._h, int(bool(on))))

    def reconstruct_raw(self, xyz_ptr: int, n: int, params: _Params):
        """Low-level call: pointer (host or device) to n x 3 f32 -> opaque surface handle."""
        out = C.c_void_p()
        _check(self._L, self._L.ss_reconstruct_surface_f32(self._h, C.c_void_p(xyz_ptr), C.c_uint64(n), C.byref(params), C.byref(out)))
        return out

    def free_surface(self, s):
        self._L.ss_surface_free(s)

    def timings(self, s) -> dict:
        t = _Timings()
        _check(self._L, self._L.ss_surface_timings(s, C.byref(t)))
        return {k: getattr(t, k) for k, _ in _Timings._fields_}


class MeshAttribute:
    """``pysplashsurf.MeshAttribute``: a named per-vertex / per-cell array (name, data, dtype).  The mesh containers of this package keep
    their attributes in plain dicts (name -> array), like ``MeshWithData.point_attributes`` of the reference returns them."""

    def __init__(self, name: str, data):
        self._name, self._data = str(name), np.asarray(data)

    @property
    def name(self) -> str:
        return self._name

    @property
    def data(self) -> np.ndarray:
        return self._data

    @property
    def dtype(self):
        return self._data.dtype


def run_splashsurf(args) -> None:
    """``pysplashsurf.run_splashsurf``: the command line of this package (`python -m splashsurf_b200`: `reconstruct`, `convert`) with an
    argv-style list whose first element is the program name.  Raises RuntimeError when the command fails, like the reference binding."""
    from .__main__ import main
    try:
        rc = main(list(args)[1:])
    except SystemExit as e:                     # argparse: unknown switch / missing argument
        rc = e.code if isinstance(e.code, int) else 1
    except (ValueError, OSError, SplashsurfError) as e:
        raise RuntimeError(str(e)) from e
    if rc:
        raise RuntimeError(f"splashsurf_b200 {' '.join(str(a) for a in list(args)[1:2])} failed (exit code {rc})")


def run_pysplashsurf() -> None:
    """Console entry point of the reference package (pysplashsurf/__init__.py:6-7)."""
    import sys
    run_splashsurf(sys.argv)


def marching_cubes(values, *, iso_surface_threshold: float, cube_size: float, translation=None, return_grid: bool = False,
                   context: Optional["Context"] = None):
    """``pysplashsurf.marching_cubes`` (pysplashsurf/src/marching_cubes.rs:108-177 -> marching_cubes::triangulate_density_map) on the GPU:
    triangulates a dense 3-D float32 array of level-set values; point (i, j, k) sits at ``translation + (i, j, k) * cube_size``, values
    above the threshold are inside (like a density).  Returns a TriMesh3d (and the UniformGrid with ``return_grid``).

    The array is cut into the 65^3-point tiles of the reconstruction's marching-cubes kernels (tiles without a sign change are skipped);
    where it does not fill whole tiles the border values are repeated, and the triangles of those padded cells -- every one of them has a
    vertex on a grid edge outside of the array -- are dropped again."""
    v = np.asarray(values)
    if v.ndim != 3:
        raise ValueError("values must be a 3D array")
    if v.dtype != np.float32:
        raise TypeError("unsupported scalar type: the device path triangulates float32 values only")
    if min(v.shape) < 2:
        raise ValueError("values needs at least two points per dimension (one cell)")
    thr, cs = np.float32(iso_surface_threshold), np.float32(cube_size)
    tr = np.zeros(3, np.float32) if translation is None else np.asarray(translation, np.float64).astype(np.float32)
    ncells = [n - 1 for n in v.shape]
    grid = UniformGrid(Aabb3d(tr.copy(), (tr + cs * np.asarray(ncells, np.float32)).astype(np.float32)), float(cs), list(v.shape), ncells)
    nt = [(c + 63) // 64 for c in ncells]
    padded = np.pad(v, [(0, t * 64 + 1 - n) for t, n in zip(nt, v.shape)], mode="edge")
    tiles, ijk = [], []
    for a in range(nt[0]):
        for b in range(nt[1]):
            for c_ in range(nt[2]):
                blk = padded[a * 64:a * 64 + 65, b * 64:b * 64 + 65, c_ * 64:c_ * 64 + 65]
                if blk.min() > thr or blk.max() < thr:        # no sign change inside this tile (NaNs compare false: kept)
                    continue
                tiles.append(blk)
                ijk.append((a, b, c_))
    ctx = default_context() if context is None else context
    L = ctx._L
    tiles = np.ascontiguousarray(np.stack(tiles)) if tiles else np.zeros((0, 65, 65, 65), np.float32)
    if len(tiles) and np.any(tiles == thr):
        # A value exactly ON the threshold is "inside" for the vertex pass (>= threshold) but for the case index only where it has a
        # neighbour below it (narrow_band_extraction.rs:79-126, :179-184).  Where the two disagree along an edge the table asks for a vertex
        # that was never created -- the reference stops with "Missing iso surface vertex at edge ..."; so does this front end (the check
        # evaluates the kernels' rules, ss_above / ss_crossing, on the tiles it is about to send).
        geq, below = tiles >= thr, tiles < thr
        nb = np.zeros_like(geq)
        for ax in (1, 2, 3):
            lo, hi = [slice(None)] * 4, [slice(None)] * 4
            lo[ax], hi[ax] = slice(0, -1), slice(1, None)
            nb[tuple(lo)] |= below[tuple(hi)]
            nb[tuple(hi)] |= below[tuple(lo)]
        above = (tiles > thr) | ((tiles == thr) & nb)
        for ax in (1, 2, 3):
            lo, hi = [slice(None)] * 4, [slice(None)] * 4
            lo[ax], hi[ax] = slice(0, -1), slice(1, None)
            if np.any((above[tuple(lo)] != above[tuple(hi)]) & (geq[tuple(lo)] == geq[tuple(hi)])):
                raise SplashsurfError(SS_ERR_INVALID_PARAMETER, "Missing iso surface vertex at an edge: a value equal to the iso-surface threshold "
                                      "lies next to a value above it without a value below it on its other side (the reference reports "
                                      "\"Missing iso surface vertex at edge ... This is a bug.\" for such an array)")
        # The reference marks such a value "above" per CELL -- only in the cells that touch one of its edges towards a value below
        # (:108-126) -- the kernels per POINT.  Where the two differ the reference either builds another mesh or stops with the error
        # above: refuse instead of returning a mesh the reference would not return.
        eq = tiles == thr
        for ca in (0, 1):
            for cb in (0, 1):
                for cc in (0, 1):
                    def corner(arr, a=ca, b=cb, c_=cc):
                        return arr[:, a:a + 64, b:b + 64, c_:c_ + 64]
                    in_cell_below = corner(below, 1 - ca, cb, cc) | corner(below, ca, 1 - cb, cc) | corner(below, ca, cb, 1 - cc)
                    ref_above = corner(tiles > thr) | (corner(eq) & in_cell_below)
                    if np.any(ref_above != corner(above)):
                        raise SplashsurfError(SS_ERR_UNSUPPORTED, "a value equal to the iso-surface threshold sits where the reference decides inside / "
                                              "outside per cell (narrow_band_extraction.rs:108-126): this degenerate configuration is not triangulated "
                                              "here -- move the threshold (or the values) by one ulp")
    ijk = np.ascontiguousarray(np.asarray(ijk, dtype=np.int32).reshape(-1, 3))
    s = C.c_void_p()
    _check(L, L.ss_marching_cubes_tiles_f32(ctx._h, tiles.ctypes.data if len(tiles) else None, len(tiles), ijk.ctypes.data if len(tiles) else None,
                                            (C.c_float * 3)(*[float(x) for x in tr]), C.c_float(float(cs)), C.c_float(float(thr)), C.byref(s)))
    try:
        nv, ntri = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s)
        verts, tris, keys = np.empty((nv, 3), np.float32), np.empty((ntri, 3), np.uint32), np.empty((nv, 4), np.int64)
        if nv:
            _check(L, L.ss_surface_copy_vertices(s, verts.ctypes.data))
            _check(L, L.ss_surface_copy_vertex_edge_keys(s, keys.ctypes.data))
        if ntri:
            _check(L, L.ss_surface_copy_triangles_u32(s, tris.ctypes.data))
    finally:
        L.ss_surface_free(s)
    # cells of the padding: a vertex whose grid edge has an end point beyond the array
    last = np.asarray(v.shape, np.int64) - 1
    end = keys[:, :3].copy()
    end[np.arange(nv), keys[:, 3]] += 1
    bad_v = (end > last).any(axis=1) if nv else np.zeros(0, bool)
    if bad_v.any():
        tris = tris[~bad_v[tris].any(axis=1)]
        newid = np.cumsum(~bad_v) - 1
        verts, tris = verts[~bad_v], newid[tris]
    mesh = TriMesh3d(np.ascontiguousarray(verts), np.ascontiguousarray(tris, dtype=np.uint64))
    return (mesh, grid) if return_grid else mesh


def neighborhood_search_spatial_hashing_parallel(particle_positions, domain: "Aabb3d", search_radius: float, *, context: Optional["Context"] = None) -> "NeighborhoodLists":
    """``pysplashsurf.neighborhood_search_spatial_hashing_parallel`` (neighborhood_search.rs:444-588) on the GPU: for every particle the
    indices of all other particles closer than ``search_radius`` (strictly), as NeighborhoodLists.  ``domain`` is the AABB whose lattice
    hashes the particles; a particle outside of it is an error (the reference panics).  The order inside a list is not specified by the
    reference (hash-map order); here it is cell by cell, ascending index inside a cell."""
    p = np.asarray(particle_positions)
    if p.dtype != np.float32:
        raise TypeError("unsupported scalar type: the device path searches float32 particles only")
    if p.ndim != 2 or p.shape[1] != 3:
        raise ValueError("particle_positions must have shape (N, 3)")
    p = np.ascontiguousarray(p)
    ctx = default_context() if context is None else context
    L = ctx._L
    lo = (C.c_float * 3)(*[float(np.float32(v)) for v in domain.min])
    hi = (C.c_float * 3)(*[float(np.float32(v)) for v in domain.max])
    s = C.c_void_p()
    _check(L, L.ss_neighborhood_search_f32(ctx._h, p.ctypes.data if len(p) else None, len(p), lo, hi, C.c_float(float(search_radius)), C.byref(s)))
    try:
        off = np.empty(len(p) + 1, dtype=np.uint64)
        idx = np.empty(L.ss_surface_num_neighbors(s), dtype=np.uint32)
        _check(L, L.ss_surface_copy_neighbor_lists(s, off.ctypes.data, idx.ctypes.data if len(idx) else None))
        return NeighborhoodLists(off, idx)
    finally:
        L.ss_surface_free(s)


class SphInterpolator:
    """``pysplashsurf.SphInterpolator`` (pysplashsurf/src/sph_interpolation.rs:25-260; splashsurf_lib sph_interpolation.rs:22-258) on the
    GPU: interpolation of per-particle quantities and of surface normals to arbitrary points with the cubic spline kernel.

    ``SphInterpolator(particle_positions (N, 3) f32, particle_densities (N,) f32, particle_rest_mass, compact_support_radius)``.
    The particle bins stay on the device inside a context of their own for the lifetime of the object (pass ``context=`` to share one:
    the interpolator is then only valid until the next reconstruction on that context).  Sums run in bin order instead of the reference's
    R-tree order: results agree with the reference to f32 round-off."""

    def __init__(self, particle_positions, particle_densities, particle_rest_mass: float, compact_support_radius: float, *, context: Optional["Context"] = None):
        p, rho = np.asarray(particle_positions), np.asarray(particle_densities)
        if p.dtype != np.float32 or rho.dtype != np.float32:
            raise TypeError("unsupported scalar type: the device path interpolates float32 data only")
        if p.ndim != 2 or p.shape[1] != 3 or rho.shape != (len(p),):
            raise ValueError("particle_positions must have shape (N, 3) and particle_densities shape (N,)")
        self._own = context is None
        self._ctx = Context() if context is None else context
        self._n = len(p)
        self._s = C.c_void_p()
        p, rho = np.ascontiguousarray(p), np.ascontiguousarray(rho)
        L = self._ctx._L
        try:
            _check(L, L.ss_sph_interpolator_create_f32(self._ctx._h, p.ctypes.data if len(p) else None, len(p), rho.ctypes.data if len(p) else None,
                                                       C.c_float(float(particle_rest_mass)), C.c_float(float(compact_support_radius)), C.byref(self._s)))
        except Exception:
            if self._own:
                self._ctx.close()
            raise

    @staticmethod
    def _points(interpolation_points) -> np.ndarray:
        x = np.asarray(interpolation_points)
        if x.dtype != np.float32:
            raise TypeError("unsupported scalar type: the device path interpolates float32 data only")
        if x.ndim != 2 or x.shape[1] != 3:
            raise ValueError("interpolation_points must have shape (M, 3)")
        return np.ascontiguousarray(x)

    def interpolate_quantity(self, particle_quantity, interpolation_points, *, first_order_correction: bool = False) -> np.ndarray:
        """Interpolates a scalar (N,) or vectorial (N, 3) per-particle quantity to the given points: (M,) or (M, 3)."""
        q, x = np.asarray(particle_quantity), self._points(interpolation_points)
        if q.dtype != np.float32:
            raise TypeError("unsupported scalar type: the device path interpolates float32 data only")
        if not ((q.ndim == 1 or (q.ndim == 2 and q.shape[1] == 3)) and len(q) == self._n):
            raise ValueError("particle_quantity must have shape (N,) or (N, 3) with one entry per particle")
        dim = 1 if q.ndim == 1 else 3
        q = np.ascontiguousarray(q)
        out = np.empty((len(x),) if dim == 1 else (len(x), 3), dtype=np.float32)
        L = self._ctx._L
        _check(L, L.ss_sph_interpolate_quantity_at_f32(self._s, q.ctypes.data if self._n else None, dim, x.ctypes.data if len(x) else None, len(x),
                                                       int(bool(first_order_correction)), out.ctypes.data if len(x) else None))
        return out

    def interpolate_normals(self, interpolation_points) -> np.ndarray:
        """Surface normals (normalised SPH gradient of the indicator function) at the given points: (M, 3)."""
        x = self._points(interpolation_points)
        out = np.empty((len(x), 3), dtype=np.float32)
        L = self._ctx._L
        _check(L, L.ss_sph_interpolate_normals_at_f32(self._s, x.ctypes.data if len(x) else None, len(x), out.ctypes.data if len(x) else None))
        return out

    def close(self):
        if getattr(self, "_s", None):
            self._ctx._L.ss_surface_free(self._s)
            self._s = None
            if self._own:
                self._ctx.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_DEFAULT_CTX: dict = {}


def default_context(device: int = -1) -> Context:
    if device not in _DEFAULT_CTX:
        _DEFAULT_CTX[device] = Context(device)
    return _DEFAULT_CTX[device]


def make_params(*, particle_radius, rest_density=1000.0, smoothing_length, cube_size, iso_surface_threshold=0.6,
                aabb_min=None, aabb_max=None, multi_threading=True, simd=True, global_neighborhood_list=False,
                subdomain_grid=True, subdomain_grid_auto_disable=True, subdomain_num_cubes_per_dim=64) -> _Params:
    """Front-end parameter mapping of pysplashsurf (reconstruction.rs:160-184): f64 products, then f32."""
    p = _Params()
    r = float(particle_radius)
    p.particle_radius = float(np.float32(r))
    p.rest_density = float(np.float32(rest_density))
    p.compact_support_radius = float(np.float32(2.0 * float(smoothing_length) * r))
    p.cube_size = float(np.float32(float(cube_size) * r))
    p.iso_surface_threshold = float(np.float32(iso_surface_threshold))
    has = aabb_min is not None and aabb_max is not None
    p.has_particle_aabb = int(has)
    if has:
        p.particle_aabb_min = (C.c_float * 3)(*[float(np.float32(v)) for v in aabb_min])
        p.particle_aabb_max = (C.c_float * 3)(*[float(np.float32(v)) for v in aabb_max])
    p.enable_multi_threading = int(bool(multi_threading))
    p.enable_simd = int(bool(simd))
    p.spatial_decomposition = int(bool(subdomain_grid))
    p.subdomain_num_cubes_per_dim = int(subdomain_num_cubes_per_dim)
    p.auto_disable = int(bool(subdomain_grid_auto_disable))
    p.global_neighborhood_list = int(bool(global_neighborhood_list))
    return p


def reconstruct_surface(particles, *, particle_radius: float, rest_density: float = 1000.0, smoothing_length: float,
                        cube_size: float, iso_surface_threshold: float = 0.6,
                        aabb_min: Optional[Sequence[float]] = None, aabb_max: Optional[Sequence[float]] = None,
                        multi_threading: bool = True, simd: bool = True, global_neighborhood_list: bool = False,
                        subdomain_grid: bool = True, subdomain_grid_auto_disable: bool = True,
                        subdomain_num_cubes_per_dim: int = 64, context: Optional[Context] = None,
                        keep_levelset_tile_of: Optional[int] = None, with_debug: bool = False, sph_normals: bool = False,
                        anisotropic: bool = False, anisotropy_max_ratio: float = 4.0, anisotropy_min_neighbors: int = 10,
                        anisotropy_smoothing: float = 0.9) -> SurfaceReconstruction:
    """Performs a surface reconstruction from the given particles (no post-processing) on the GPU.

    Same signature and semantics as ``pysplashsurf.reconstruct_surface``; ``particles`` is an (N, 3) float32
    array (float64 input is not provided by the device path and raises, like an unsupported dtype does in the
    reference, pysplashsurf/src/reconstruction.rs:204-206).

    ``anisotropic=True`` (an extension of the device path) splats anisotropic kernels (Yu & Turk 2013): every kernel is
    stretched along the principal axes of its neighbourhood (radii in [R / anisotropy_max_ratio, R], isotropic below
    ``anisotropy_min_neighbors`` neighbours) and centred at the particle moved by ``anisotropy_smoothing`` times the weighted mean
    offset of its neighbours.  Thin sheets come out thinner and flat surfaces smoother.  ``with_debug`` then also returns the
    per-particle ``anisotropic_centers``, ``anisotropic_matrices`` and ``anisotropic_factors``.  SPH normals are the gradient of
    the isotropic field and cannot be combined with it.
    """
    if anisotropic and sph_normals:
        raise ValueError("sph_normals are the gradient of the isotropic field: not available with anisotropic=True")
    arr = np.asarray(particles)
    if arr.dtype != np.float32:
        raise TypeError("unsupported scalar type: the device path reconstructs float32 particles only")
    if arr.ndim != 2 or arr.shape[1] != 3:
        raise ValueError("particles must have shape (N, 3)")
    arr = np.ascontiguousarray(arr)
    ctx = context or default_context()
    L = ctx._L
    p = make_params(particle_radius=particle_radius, rest_density=rest_density, smoothing_length=smoothing_length,
                    cube_size=cube_size, iso_surface_threshold=iso_surface_threshold, aabb_min=aabb_min, aabb_max=aabb_max,
                    multi_threading=multi_threading, simd=simd, global_neighborhood_list=global_neighborhood_list,
                    subdomain_grid=subdomain_grid, subdomain_grid_auto_disable=subdomain_grid_auto_disable,
                    subdomain_num_cubes_per_dim=subdomain_num_cubes_per_dim)
    _check(L, L.ss_context_keep_levelset_tile(ctx._h, -1 if keep_levelset_tile_of is None else int(keep_levelset_tile_of)))
    _check(L, L.ss_context_set_compute_sph_normals(ctx._h, int(bool(sph_normals))))
    try:
        _set_anisotropy(ctx, anisotropic, anisotropy_max_ratio, anisotropy_min_neighbors, anisotropy_smoothing)
        s = ctx.reconstruct_raw(arr.ctypes.data, len(arr), p)
    except BaseException:
        _check(L, L.ss_context_set_compute_sph_normals(ctx._h, 0))
        _check(L, L.ss_context_set_anisotropy_f32(ctx._h, None))
        raise
    try:
        res = _collect(ctx, s, len(arr), p, with_debug or keep_levelset_tile_of is not None, keep_levelset_tile_of is not None)
        if sph_normals:
            nrm = np.empty((res.mesh.nvertices, 3), dtype=np.float32)
            if len(nrm):
                _check(L, L.ss_surface_copy_normals(s, nrm.ctypes.data))
            res.normals = nrm
        if anisotropic:
            _collect_anisotropy(ctx, s, res, with_debug)
        return res
    finally:
        _check(L, L.ss_context_set_compute_sph_normals(ctx._h, 0))
        _check(L, L.ss_context_set_anisotropy_f32(ctx._h, None))
        ctx.free_surface(s)


def _set_anisotropy(ctx: Context, anisotropic: bool, max_ratio: float, min_neighbors: int, smoothing: float) -> None:
    """Switches the context's anisotropic kernels on (with these parameters) or off; the caller resets it after the call."""
    if not anisotropic:
        _check(ctx._L, ctx._L.ss_context_set_anisotropy_f32(ctx._h, None))
        return
    if int(min_neighbors) != min_neighbors or not 0 <= int(min_neighbors) < 2 ** 32:
        raise ValueError("anisotropy_min_neighbors must be a non-negative integer")
    a = _Anisotropy(float(np.float32(max_ratio)), int(min_neighbors), float(np.float32(smoothing)))
    _check(ctx._L, ctx._L.ss_context_set_anisotropy_f32(ctx._h, C.byref(a)))


def _collect_anisotropy(ctx: Context, s, res: SurfaceReconstruction, debug: bool) -> None:
    L = ctx._L
    ms, sweeps = (C.c_float * 2)(), C.c_uint32()
    _check(L, L.ss_surface_anisotropy_stats(s, ms, C.byref(sweeps)))
    res.timings.update(anisotropy_moments=ms[0], anisotropy_decomposition=ms[1], anisotropy_max_jacobi_sweeps=sweeps.value)
    if debug:
        n = L.ss_surface_num_particles(s)
        res.anisotropic_centers = np.empty((n, 3), np.float32)
        res.anisotropic_matrices = np.empty((n, 6), np.float32)
        res.anisotropic_factors = np.empty(n, np.float32)
        _check(L, L.ss_surface_copy_anisotropy_f32(s, res.anisotropic_centers.ctypes.data, res.anisotropic_matrices.ctypes.data,
                                                   res.anisotropic_factors.ctypes.data))


def _collect(ctx: Context, s, n_in: int, p: _Params, debug: bool, tile: bool) -> SurfaceReconstruction:
    L = ctx._L
    nv, nt, n = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s), L.ss_surface_num_particles(s)
    if getattr(ctx, "reuse_host_buffers", False):
        # opt-in: the big result arrays are views of page-locked buffers of the context, overwritten by its next reconstruction
        verts, tris, dens = ctx.host_array("vertices", (nv, 3), np.float32), ctx.host_array("triangles", (nt, 3), np.uint64), ctx.host_array("densities", (n,), np.float32)
    else:
        verts = np.empty((nv, 3), dtype=np.float32)
        tris = np.empty((nt, 3), dtype=np.uint64)
        dens = np.empty(n, dtype=np.float32)
    _check(L, L.ss_surface_copy_vertices(s, verts.ctypes.data))
    _check(L, L.ss_surface_copy_triangles_u64(s, tris.ctypes.data))
    _check(L, L.ss_surface_copy_particle_densities(s, dens.ctypes.data))
    g = _Grid()
    _check(L, L.ss_surface_grid(s, C.byref(g)))
    sub = None
    if L.ss_surface_used_decomposition(s):
        sg = _Grid()
        _check(L, L.ss_surface_subdomain_grid(s, C.byref(sg)))
        sub = UniformGrid._from(sg)
    inside = None
    if p.has_particle_aabb:
        inside = np.empty(n_in, dtype=np.uint8)
        if n_in:
            _check(L, L.ss_surface_copy_particle_inside_aabb(s, inside.ctypes.data))
        inside = inside.astype(bool)
    res = SurfaceReconstruction(mesh=TriMesh3d(verts, tris), grid=UniformGrid._from(g), subdomain_grid=sub,
                                particle_densities=dens, particle_inside_aabb=inside, timings=ctx.timings(s))
    if p.global_neighborhood_list:
        off = np.empty(n + 1, dtype=np.uint64)
        idx = np.empty(L.ss_surface_num_neighbors(s), dtype=np.uint32)
        _check(L, L.ss_surface_copy_neighbor_lists(s, off.ctypes.data, idx.ctypes.data if len(idx) else None))
        res.particle_neighbors = NeighborhoodLists(off, idx)
    if debug:
        keys = np.empty((nv, 4), dtype=np.int64)
        _check(L, L.ss_surface_copy_vertex_edge_keys(s, keys.ctypes.data))
        res.vertex_edge_keys = keys
        ns = L.ss_surface_num_subdomains(s)
        flat, cnt, sp = np.empty(ns, np.int64), np.empty(ns, np.uint64), np.empty(ns, np.uint8)
        _check(L, L.ss_surface_copy_subdomains(s, flat.ctypes.data, cnt.ctypes.data, sp.ctypes.data))
        res.subdomains = {"flat": flat, "count": cnt, "sparse": sp.astype(bool)}
    if tile:
        S = int(p.subdomain_num_cubes_per_dim)
        t = np.empty((S + 1,) * 3, dtype=np.float32)
        _check(L, L.ss_surface_copy_levelset_tile(s, t.ctypes.data))
        res.levelset_tile = t
    return res


def density_grid_loop(subdomain_particles, subdomain_particle_densities, *, global_min, cube_size, subdomain_ijk,
                      subdomain_cubes: int, compact_support_radius: float, particle_rest_mass: float, simd: bool = True,
                      context: Optional[Context] = None) -> np.ndarray:
    """Level-set tile of one subdomain: the device counterpart of ``density_grid_loop_auto`` (simd=True) /
    ``density_grid_loop_scalar`` (simd=False), splashsurf_lib/src/dense_subdomains.rs:715-847.
    Returns the (S+1, S+1, S+1) float32 tile."""
    ctx = context or default_context()
    L = ctx._L
    xyz = np.ascontiguousarray(subdomain_particles, dtype=np.float32).reshape(-1, 3)
    rho = np.ascontiguousarray(subdomain_particle_densities, dtype=np.float32)
    if len(rho) != len(xyz):
        raise ValueError("one density per particle is required")
    gmin = np.ascontiguousarray(global_min, dtype=np.float32)
    sijk = np.ascontiguousarray(subdomain_ijk, dtype=np.int64)
    S = int(subdomain_cubes)
    out = np.empty((S + 1,) * 3, dtype=np.float32)
    _check(L, L.ss_levelset_tile_f32(ctx._h, xyz.ctypes.data, rho.ctypes.data, len(xyz), gmin.ctypes.data,
                                     C.c_float(float(np.float32(cube_size))), sijk.ctypes.data, S,
                                     C.c_float(float(np.float32(compact_support_radius))),
                                     C.c_float(float(np.float32(particle_rest_mass))), 0 if simd else 1, out.ctypes.data))
    return out


class MeshType(Enum):
    """pysplashsurf.MeshType: the kind of mesh a MeshWithData wraps."""
    Tri3d = 0
    MixedTriQuad3d = 1


@dataclass
class MeshWithData:
    """Mirrors pysplashsurf.MeshWithData for the attributes this package can produce."""
    mesh: TriMesh3d
    point_attributes: dict = field(default_factory=dict)
    cell_attributes: dict = field(default_factory=dict)

    def __post_init__(self):
        if not isinstance(self.mesh, (TriMesh3d, MixedTriQuadMesh3d)):
            raise TypeError("unsupported mesh type, expected TriMesh3d or MixedTriQuadMesh3d")

    @property
    def nvertices(self) -> int:
        return self.mesh.nvertices

    @property
    def ncells(self) -> int:
        return self.mesh.ncells

    @property
    def dtype(self):
        return np.dtype(np.float32)

    @property
    def mesh_type(self) -> "MeshType":
        return MeshType.MixedTriQuad3d if isinstance(self.mesh, MixedTriQuadMesh3d) else MeshType.Tri3d

    def copy_mesh(self):
        return self.mesh.copy()

    def copy(self) -> "MeshWithData":
        return MeshWithData(self.mesh.copy(), {k: np.array(v) for k, v in self.point_attributes.items()},
                            {k: np.array(v) for k, v in self.cell_attributes.items()})

    @staticmethod
    def _attribute(attribute, n: int, what: str) -> np.ndarray:
        """pysplashsurf/src/mesh.rs add_*_attribute: uint64 (N,), float32 (N,) or float32 (N, 3); the data is copied."""
        a = np.asarray(attribute)
        if a.dtype not in (np.dtype(np.uint64), np.dtype(np.float32)):
            raise TypeError("unsupported attribute data type")
        if not (a.ndim == 1 or (a.ndim == 2 and a.shape[1] in (1, 3))) or (a.ndim == 2 and a.dtype != np.float32):
            raise ValueError("expected Nx1 or Nx3 array for Vector3Real attribute data")
        if len(a) != n:
            raise ValueError(f"number of attribute values must match number of {what} in the mesh")
        return np.ascontiguousarray(a.reshape(-1) if a.ndim == 2 and a.shape[1] == 1 else a).copy()

    def add_point_attribute(self, name: str, attribute) -> None:
        self.point_attributes[str(name)] = self._attribute(attribute, self.nvertices, "vertices")

    def add_cell_attribute(self, name: str, attribute) -> None:
        self.cell_attributes[str(name)] = self._attribute(attribute, self.ncells, "cells")

    def write_to_file(self, path, *, file_format: Optional[str] = None) -> None:
        """``pysplashsurf.MeshWithData.write_to_file``; the file is the one the reference CLI writes for this mesh (`write_mesh`)."""
        write_mesh(path, self, file_format=file_format)


_MESH_FORMATS = {None: 0, "vtk": 1, "vtk42": 1, "ply": 2, "obj": 3}


def write_mesh(path, mesh, *, point_attributes: Optional[dict] = None, cell_attributes: Optional[dict] = None, file_format: Optional[str] = None,
               threads: int = 0) -> None:
    """``splashsurf::io::write_mesh`` (splashsurf/src/io.rs:276-316): writes a TriMesh3d, MixedTriQuadMesh3d, MeshWithData or a
    ``(vertices, triangles)`` pair to ``.vtk`` (legacy binary), ``.ply`` (binary little endian) or ``.obj``, picked by the extension
    unless ``file_format`` names one.  Native multi-threaded writer (ss_write_mesh_f32); the bytes are those of the reference CLI's file
    for the same mesh and attributes (float32 scalars / 3-vectors and uint64 scalars; a point attribute called "normals" becomes the
    vn lines of an OBJ and nx / ny / nz of a PLY)."""
    if hasattr(mesh, "point_attributes"):
        point_attributes = {**mesh.point_attributes, **(point_attributes or {})}
        cell_attributes = {**mesh.cell_attributes, **(cell_attributes or {})}
        mesh = mesh.mesh
    if isinstance(mesh, tuple):
        verts, tris, quads = mesh[0], mesh[1], (mesh[2] if len(mesh) > 2 else None)
    elif isinstance(mesh, MixedTriQuadMesh3d):
        verts, tris, quads = mesh.vertices, mesh.get_triangles(), mesh.get_quads()
    else:
        verts, tris, quads = mesh.vertices, mesh.triangles, None
    if file_format not in _MESH_FORMATS:
        raise ValueError(f"unsupported mesh file format {file_format!r}")
    L = load_library()
    v = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3)
    t = np.asarray(tris)
    idt = np.uint32 if t.dtype.itemsize == 4 and t.dtype.kind in "ui" else np.uint64
    t = np.ascontiguousarray(t, dtype=idt).reshape(-1, 3)
    q = np.ascontiguousarray(quads if quads is not None else np.zeros((0, 4)), dtype=idt).reshape(-1, 4)
    if len(t) and int(t.max()) >= len(v) or len(q) and int(q.max()) >= len(v):
        raise ValueError("cell refers to a vertex that does not exist")
    keep = []

    def table(attrs, n, what):
        arr = (_MeshAttribute * max(1, len(attrs or {})))()
        for i, (name, a) in enumerate((attrs or {}).items()):
            a = np.asarray(a)
            if a.dtype.kind in "ui" and a.ndim == 1:
                a, kind = np.ascontiguousarray(a, dtype=np.uint64), 2
            elif a.ndim == 1:
                a, kind = np.ascontiguousarray(a, dtype=np.float32), 0
            elif a.ndim == 2 and a.shape[1] == 3:
                a, kind = np.ascontiguousarray(a, dtype=np.float32), 1
            else:
                raise ValueError(f"{what} attribute {name!r}: expected shape (n,) or (n, 3)")
            if len(a) != n:
                raise ValueError(f"{what} attribute {name!r} has {len(a)} entries for {n} {what}s")
            keep.append(a)
            nm = str(name).encode()
            keep.append(nm)
            arr[i] = _MeshAttribute(nm, kind, a.ctypes.data if len(a) else None)
        return arr, len(attrs or {})
    pa, npa = table(point_attributes, len(v), "point")
    ca, nca = table(cell_attributes, len(t) + len(q), "cell")
    _check(L, L.ss_write_mesh_f32(os.fspath(path).encode(), _MESH_FORMATS[file_format], v.ctypes.data if len(v) else None, len(v),
                                  t.ctypes.data if len(t) else None, len(t), q.ctypes.data if len(q) else None, len(q), t.dtype.itemsize,
                                  pa, npa, ca, nca, int(threads)))


def reconstruction_pipeline(particles, *, attributes_to_interpolate=None, particle_radius: float, rest_density: float = 1000.0,
                            smoothing_length: float, cube_size: float, iso_surface_threshold: float = 0.6, aabb_min=None, aabb_max=None,
                            multi_threading: bool = True, simd: bool = True, subdomain_grid: bool = True,
                            subdomain_grid_auto_disable: bool = True, subdomain_num_cubes_per_dim: int = 64,
                            compute_normals: bool = False, sph_normals: bool = False, normals_smoothing_iters: Optional[int] = None,
                            mesh_smoothing_iters: Optional[int] = None, mesh_smoothing_weights: bool = True,
                            mesh_smoothing_weights_normalization: float = 13.0, output_mesh_smoothing_weights: bool = False,
                            output_raw_normals: bool = False, output_raw_mesh: bool = False, context: Optional[Context] = None,
                            with_debug: bool = False, anisotropic: bool = False, anisotropy_max_ratio: float = 4.0,
                            anisotropy_min_neighbors: int = 10, anisotropy_smoothing: float = 0.9, **post):
    """``pysplashsurf.reconstruction_pipeline`` (pysplashsurf/src/pipeline.rs:109-200) on the GPU: surface reconstruction plus
    the post-processing steps of splashsurf/src/reconstruct.rs:1094-1391 that run on the device -- smoothing weights, weighted
    Laplacian smoothing, SPH or area-weighted normals (at the smoothed vertices), normal smoothing and SPH interpolation of
    float32 particle attributes.  Returns ``(MeshWithData, SurfaceReconstruction)``; the reconstruction holds the raw mesh.

    ``mesh_cleanup`` (+ ``mesh_cleanup_snap_dist``, 5 sweeps) and ``decimate_barnacles`` (+ ``keep_vertices``) run first, as in
    reconstruct.rs:1058-1092 -- sequential half-edge collapses on the host (library entries ss_mesh_cleanup_f32 /
    ss_mesh_decimation_f32), after which the new mesh goes back to the device for the remaining steps.  ``generate_quads`` (+
    ``quad_max_edge_diag_ratio`` / ``quad_max_normal_angle`` / ``quad_max_interior_angle``) runs last (reconstruct.rs:1410-1441, host):
    the returned mesh is then a MixedTriQuadMesh3d.  ``mesh_aabb_min`` / ``mesh_aabb_max`` (+ ``mesh_aabb_clamp_vertices``) clamp the
    finished mesh (reconstruct.rs:1394-1408) and ``check_mesh_closed`` / ``check_mesh_manifold`` raise SplashsurfError with the
    reference's message when the check fails (:1445-1470); ``check_mesh_orientation`` likewise (:1481-1541).

    ``anisotropic`` and the ``anisotropy_*`` parameters select anisotropic kernels as in ``reconstruct_surface``; every step above then
    runs on the anisotropic mesh (attribute interpolation still sums over the particles' isotropic kernels), except SPH normals."""
    if anisotropic and sph_normals:
        raise ValueError("sph_normals are the gradient of the isotropic field: not available with anisotropic=True")
    passive = ("mesh_cleanup", "decimate_barnacles", "mesh_cleanup_snap_dist", "keep_vertices", "generate_quads", "quad_max_edge_diag_ratio",
               "quad_max_normal_angle", "quad_max_interior_angle", "mesh_aabb_min", "mesh_aabb_max", "mesh_aabb_clamp_vertices",
               "check_mesh_closed", "check_mesh_manifold", "check_mesh_orientation", "check_mesh_debug")
    enabled = [k for k, v in post.items() if v not in (False, None, 0) and k not in passive]
    if enabled:
        raise NotImplementedError(f"post-processing not provided by the device path: {enabled}")
    mesh_cleanup, decimate_barnacles = bool(post.get("mesh_cleanup", False)), bool(post.get("decimate_barnacles", False))
    keep_vertices, snap_dist = bool(post.get("keep_vertices", False)), post.get("mesh_cleanup_snap_dist", None)
    arr = np.asarray(particles)
    if arr.dtype != np.float32:
        raise TypeError("unsupported scalar type: the device path reconstructs float32 particles only")
    if arr.ndim != 2 or arr.shape[1] != 3:
        raise ValueError("particles must have shape (N, 3)")
    arr = np.ascontiguousarray(arr)
    attributes = {}
    for name, a in (attributes_to_interpolate or {}).items():
        a = np.asarray(a)
        if a.dtype != np.float32 or not (a.ndim == 1 or (a.ndim == 2 and a.shape[1] == 3)) or len(a) != len(arr):
            raise NotImplementedError(f"attribute {name!r}: only float32 arrays of shape (N,) or (N, 3) are interpolated")
        attributes[name] = np.ascontiguousarray(a)
    ctx = context or default_context()
    L = ctx._L
    p = make_params(particle_radius=particle_radius, rest_density=rest_density, smoothing_length=smoothing_length, cube_size=cube_size,
                    iso_surface_threshold=iso_surface_threshold, aabb_min=aabb_min, aabb_max=aabb_max, multi_threading=multi_threading,
                    simd=simd, subdomain_grid=subdomain_grid, subdomain_grid_auto_disable=subdomain_grid_auto_disable,
                    subdomain_num_cubes_per_dim=subdomain_num_cubes_per_dim)
    _check(L, L.ss_context_keep_levelset_tile(ctx._h, -1))
    _check(L, L.ss_context_set_compute_sph_normals(ctx._h, 0))
    try:
        _set_anisotropy(ctx, anisotropic, anisotropy_max_ratio, anisotropy_min_neighbors, anisotropy_smoothing)
        s = ctx.reconstruct_raw(arr.ctypes.data, len(arr), p)
    finally:
        _check(L, L.ss_context_set_anisotropy_f32(ctx._h, None))
    try:
        rec = _collect(ctx, s, len(arr), p, with_debug, False)                  # raw mesh, densities, grids
        if anisotropic:
            _collect_anisotropy(ctx, s, rec, with_debug)
        out_mesh = rec.mesh
        if mesh_cleanup or decimate_barnacles:                                  # reconstruct.rs:1058-1092
            out_mesh = rec.mesh.copy()
            if mesh_cleanup:
                marching_cubes_cleanup(out_mesh, rec.grid, max_rel_snap_dist=snap_dist, max_iter=5, keep_vertices=keep_vertices)
            if decimate_barnacles:
                barnacle_decimation(out_mesh, keep_vertices=keep_vertices)
            t32 = np.ascontiguousarray(out_mesh.triangles, dtype=np.uint32)
            _check(L, L.ss_surface_replace_mesh_f32(s, out_mesh.vertices.ctypes.data if out_mesh.nvertices else None, out_mesh.nvertices,
                                                    t32.ctypes.data if len(t32) else None, len(t32)))
        nv = out_mesh.nvertices
        point = {}
        weights_used = bool(mesh_smoothing_weights)
        if weights_used:                                                        # reconstruct.rs:1159-1258 (at the raw vertices)
            wnn, sw = np.empty(nv, np.float32), np.empty(nv, np.float32)
            _check(L, L.ss_surface_compute_smoothing_weights_f32(s, C.c_float(float(np.float32(mesh_smoothing_weights_normalization))),
                                                                 wnn.ctypes.data if nv else None, sw.ctypes.data if nv else None))
            if output_mesh_smoothing_weights:
                point["wnn"], point["sw"] = wnn, sw
        if mesh_smoothing_iters is not None:                                    # reconstruct.rs:1261-1279, beta = 1
            _check(L, L.ss_surface_laplacian_smoothing_f32(s, int(mesh_smoothing_iters), C.c_float(1.0), None))
        verts = out_mesh.vertices
        if mesh_smoothing_iters:
            verts = np.empty((nv, 3), np.float32)
            _check(L, L.ss_surface_copy_vertices(s, verts.ctypes.data))
        if compute_normals:                                                     # reconstruct.rs:1282-1342
            _check(L, L.ss_surface_compute_normals_f32(s, int(bool(sph_normals))))
            raw = np.empty((nv, 3), np.float32)
            if nv:
                _check(L, L.ss_surface_copy_normals(s, raw.ctypes.data))
            if normals_smoothing_iters is not None:
                _check(L, L.ss_surface_smooth_normals_f32(s, int(normals_smoothing_iters)))
                sm = np.empty((nv, 3), np.float32)
                if nv:
                    _check(L, L.ss_surface_copy_normals(s, sm.ctypes.data))
                point["normals"] = sm
                if output_raw_normals:
                    point["raw_normals"] = raw
            else:
                point["normals"] = raw
        inside = rec.particle_inside_aabb
        for name, a in attributes.items():                                      # reconstruct.rs:1345-1391 (filtered_quantity)
            vals = np.ascontiguousarray(a[inside]) if inside is not None else a
            dim = 1 if vals.ndim == 1 else 3
            out = np.empty(nv if dim == 1 else (nv, 3), np.float32)
            _check(L, L.ss_surface_interpolate_quantity_f32(s, vals.ctypes.data if len(vals) else None, dim, 1, out.ctypes.data if nv else None))
            point[name] = out
        rec.normals = point.get("normals")
        mesh = TriMesh3d(verts, out_mesh.triangles)
        if post.get("mesh_aabb_min") is not None and post.get("mesh_aabb_max") is not None:     # reconstruct.rs:1394-1408
            mesh, point = clamp_mesh_with_aabb(mesh, post["mesh_aabb_min"], post["mesh_aabb_max"], clamp_vertices=bool(post.get("mesh_aabb_clamp_vertices", True)),
                                               keep_vertices=keep_vertices, point_attributes=point)
        if (post.get("check_mesh_closed") or post.get("check_mesh_manifold")) and not post.get("generate_quads", False):   # :1445-1470
            problems = check_mesh_consistency(mesh, rec.grid, check_closed=bool(post.get("check_mesh_closed")),
                                              check_manifold=bool(post.get("check_mesh_manifold")), debug=bool(post.get("check_mesh_debug")))
            if problems:
                raise SplashsurfError(SS_ERR_MESH_CHECK, problems)
        if post.get("check_mesh_orientation") and not post.get("generate_quads", False):          # reconstruct.rs:1481-1541
            flipped = find_flipped_faces(mesh)
            if len(flipped):
                raise SplashsurfError(SS_ERR_MESH_CHECK, f"Mesh is not consistently oriented. Found {len(flipped)} faces with normals flipped relative to adjacent vertices.")
        if post.get("generate_quads", False):                                  # reconstruct.rs:1410-1441
            mesh = convert_tris_to_quads(mesh, non_squareness_limit=post.get("quad_max_edge_diag_ratio", 1.75),
                                         normal_angle_limit=post.get("quad_max_normal_angle", 10.0),
                                         max_interior_angle=post.get("quad_max_interior_angle", 135.0))
        return MeshWithData(mesh, point, {}), rec
    finally:
        ctx.free_surface(s)
