"""CPU tests of the drop-in boundary: the C-ABI library builds, loads, exports every symbol the header declares,
and refuses to run without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "splashsurf_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(ss_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol(ss):
    L = ss.load_library()
    names = declared_symbols()
    assert "ss_reconstruct_surface_f32" in names and "ss_levelset_tile_f32" in names and len(names) >= 25
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/splashsurf_b200.h but not exported"
    assert L.ss_abi_version() == 3


def test_params_struct_layout_matches_header(ss):
    # 5 floats, i32, 2x3 floats, 3 x i32, u32, 2 x i32  = 68 bytes, no padding
    assert C.sizeof(ss._Params) == 4 * (5 + 1 + 6 + 3 + 1 + 2)
    assert C.sizeof(ss._Grid) == 4 * 7 + 4 + 8 * 6     # 7 floats (+4 pad) + 6 int64


def test_no_cpu_fallback_without_gpu(ss):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ss.SplashsurfError) as e:
        ss.Context()
    assert e.value.code == 101          # SS_ERR_NO_DEVICE
    with pytest.raises(ss.SplashsurfError):
        ss.reconstruct_surface(np.zeros((4, 3), np.float32), particle_radius=0.025, smoothing_length=2.0, cube_size=0.5)


def test_front_end_parameter_mapping(ss):
    """pysplashsurf multiplies smoothing_length and cube_size by the particle radius in f64, then casts to f32
    (pysplashsurf/src/reconstruction.rs:172-176)."""
    p = ss.make_params(particle_radius=0.025, smoothing_length=2.2, cube_size=1.1)
    assert p.compact_support_radius == float(np.float32(2.0 * 2.2 * 0.025))
    assert p.cube_size == float(np.float32(1.1 * 0.025))
    assert p.spatial_decomposition == 1 and p.auto_disable == 1 and p.subdomain_num_cubes_per_dim == 64
    with pytest.raises(TypeError):
        ss.reconstruct_surface(np.zeros((4, 3), np.float64), particle_radius=0.025, smoothing_length=2.0, cube_size=0.5)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "splashsurf_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "liboracle" not in src, f


def test_ctypes_signatures_match_header_arity(ss):
    """Every binding in splashsurf_b200/__init__.py that declares argtypes has as many arguments as the C declaration."""
    hdr = open(os.path.join(ROOT, "include", "splashsurf_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    L = ss.load_library()
    checked = 0
    for m in re.finditer(r"\b(ss_[a-z0-9_]+)\s*\(([^;{}]*?)\)\s*;", hdr, flags=re.S):
        name, args = m.group(1), m.group(2).strip()
        # drop nested parentheses of function-pointer parameters before counting commas
        flat = re.sub(r"\([^()]*\)", "", args)
        n = 0 if flat in ("", "void") else flat.count(",") + 1
        fn = getattr(L, name)
        if fn.argtypes is not None:
            assert len(fn.argtypes) == n, (name, len(fn.argtypes), n)
            checked += 1
    assert checked >= 25


def test_python_mirror_covers_the_public_names_of_pysplashsurf(ss, oracle_mod, tmp_path, reference_output):
    """Every public class / function of the reference's Python module exists under the same name here (its sub-modules aside; the
    names are stored in tests/golden/reference_outputs.json)."""
    import types

    def public_names():
        ps = oracle_mod.reference()
        return [n for n in dir(ps) if not n.startswith("_") and not isinstance(getattr(ps, n), types.ModuleType)]
    names = reference_output("pysplashsurf_public_names", public_names)
    assert len(names) >= 20 and [n for n in names if not hasattr(ss, n)] == []
    # run_splashsurf drives this package's command line (no device needed for `convert`)
    import numpy as np
    src, dst = str(tmp_path / "a.xyz"), str(tmp_path / "a.json")
    np.arange(12, dtype=np.float32).tofile(src)
    ss.run_splashsurf(["splashsurf", "convert", "--particles", src, "-o", dst])
    assert open(dst).read() == "[[0.0,1.0,2.0],[3.0,4.0,5.0],[6.0,7.0,8.0],[9.0,10.0,11.0]]"
    with pytest.raises(RuntimeError):
        ss.run_splashsurf(["splashsurf", "convert", "--particles", src, "-o", dst])          # exists, no --overwrite
    a = ss.MeshAttribute("w", np.ones(3, np.float32))
    assert (a.name, a.dtype, a.data.shape) == ("w", np.float32, (3,))


def test_cell_local_numbering_tables_of_the_kernels():
    """uniform_grid.rs:806-930 (CELL_LOCAL_POINT_COORDS, CELL_LOCAL_EDGES and their consistency tests): the corner order behind the case index
    and the (origin corner, axis) of the twelve local edges as the marching-cubes kernels hold them (csrc/ss_kernels.cuh, csrc/ss_mc.cuh)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "splashsurf_b200", "csrc", "ss_kernels.cuh")).read()
    corners = [(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)]      # CELL_LOCAL_POINT_COORDS
    edges = [(0, 0), (1, 1), (3, 0), (0, 1), (4, 0), (5, 1), (7, 0), (4, 1), (0, 2), (1, 2), (2, 2), (3, 2)]  # CELL_LOCAL_EDGES (corner, axis)
    m = re.search(r"c_edge_org\[12\]\[3\]\s*=\s*\{(.*?)\};", src, re.S)
    org = [tuple(int(x) for x in g.split(",")) for g in re.findall(r"\{([^{}]*)\}", m.group(1))]
    m = re.search(r"c_edge_axis\[12\]\s*=\s*\{(.*?)\};", src, re.S)
    axis = [int(x) for x in m.group(1).split(",")]
    assert org == [corners[c] for c, _ in edges] and axis == [a for _, a in edges]
    # the case index sets bit v for corner v in exactly this order (ss_case_index)
    body = src[src.index("__device__ __forceinline__ int ss_case_index"):]
    body = body[:body.index("return idx;")]
    seen = [tuple(int(x) for x in g) for g in re.findall(r"// corner \d \((\d),(\d),(\d)\)", body)]
    assert seen == corners
    # consistency tests of the reference: the flattened coordinate finds the corner, every edge starts at the corner with the lower coordinate
    local_points = [0, 1, 3, 2, 4, 5, 7, 6]                                                                   # CELL_LOCAL_POINTS
    for v, (x, y, z) in enumerate(corners):
        assert local_points[x + 2 * y + 4 * z] == v
    for c, a in edges:
        assert corners[c][a] == 0
