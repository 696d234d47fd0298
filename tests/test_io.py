"""CPU tests of the harness I/O helpers (SURVEY.md 8f #3) against the reference binary's own reader / writer."""
import os

import numpy as np
import pytest


def test_xyz_roundtrip_and_obj_roundtrip(tmp_path, ss):
    from splashsurf_b200 import io
    p = np.random.default_rng(0).normal(size=(257, 3)).astype(np.float32)
    io.write_xyz(str(tmp_path / "p.xyz"), p)
    assert np.array_equal(io.read_xyz(str(tmp_path / "p.xyz")), p)
    v = np.array([[0, 0, 0], [1, 0, 0.5], [0, 1e-7, 2.25]], np.float32)
    t = np.array([[0, 1, 2]])
    io.write_obj(str(tmp_path / "m.obj"), v, t)
    v2, t2 = io.read_obj(str(tmp_path / "m.obj"))
    assert np.array_equal(v2, v) and np.array_equal(t2, t)          # shortest round-trip formatting is lossless


def test_obj_and_xyz_interoperate_with_reference_cli(tmp_path, oracle_mod, ss, reference_output):
    """The reference CLI reads our .xyz and its OBJ output parses with our reader to the mesh its API returns.  Its OBJ file is stored
    as tests/golden/reference_cli_cube8.obj.gz; the .xyz it read and the size of its API mesh in tests/golden/reference_outputs.json."""
    import gzip
    from conftest import GOLDEN, digest
    from splashsurf_b200 import io, synthetic as syn
    p = syn.jittered_cube(8, 0.025, 5)
    xyz, obj = str(tmp_path / "p.xyz"), str(tmp_path / "out.obj")
    io.write_xyz(xyz, p)
    stored = os.path.join(GOLDEN, "reference_cli_cube8.obj.gz")

    def run_reference():
        ps = oracle_mod.reference()
        ps.run_splashsurf(["splashsurf", "reconstruct", xyz, "-r=0.025", "-l=2.0", "-c=0.75", "-o", obj, "-q"])
        with open(obj, "rb") as f, gzip.GzipFile(stored, "wb", mtime=0) as g:
            g.write(f.read())
        r = ps.reconstruct_surface(p, particle_radius=0.025, smoothing_length=2.0, cube_size=0.75, subdomain_grid_auto_disable=False)
        return {"xyz": digest(open(xyz, "rb").read()), "nv": len(r.mesh.vertices), "nt": len(r.mesh.triangles)}
    want = reference_output("obj_interop.cube8", run_reference)
    assert digest(open(xyz, "rb").read()) == want["xyz"]                  # the file the reference CLI read
    with gzip.open(stored) as f, open(obj, "wb") as g:
        g.write(f.read())
    v, t = io.read_obj(obj)
    assert len(v) == want["nv"] and len(t) == want["nt"]
    ours = str(tmp_path / "ours.obj")
    io.write_obj(ours, v, t)
    v2, t2 = io.read_obj(ours)
    assert np.array_equal(v2, v) and np.array_equal(t2, t)


# ---- mesh writers (csrc/ss_meshio.inc behind ss_write_mesh_f32): whole files against the reference CLI's -------------------------------
def _rewrite_and_compare(ss, ply_path, stem, tmp_path, threads, digests=None):
    """Reads the reference's .ply (it holds every value of the mesh), writes .vtk / .ply / .obj with the library, compares whole files
    (with the reference's files <stem>.<ext>, or with their digests {ext: digest})."""
    from conftest import digest
    from splashsurf_b200 import io
    v, t, q, attrs = io.read_ply_mesh(ply_path)
    mesh = ss.MixedTriQuadMesh3d(v, t.astype(np.uint64), q.astype(np.uint64)) if len(q) else ss.TriMesh3d(v, t.astype(np.uint64))
    mwd = ss.MeshWithData(mesh, attrs, {})
    for ext in ("vtk", "ply", "obj"):
        out = str(tmp_path / f"out_{threads}.{ext}")
        ss.write_mesh(out, mwd, threads=threads)
        if digests is None:
            assert open(out, "rb").read() == open(f"{stem}.{ext}", "rb").read(), (stem, ext, threads)
        else:
            assert digest(open(out, "rb").read()) == digests[ext], (stem, ext, threads)
    return v, t, q, attrs


@pytest.mark.parametrize("case", ["attr", "quad"])
def test_mesh_writers_reproduce_reference_files(ss, tmp_path, case):
    """tests/golden/meshio_*.{vtk,ply,obj} were written by the reference CLI (tools/make_golden_meshio.py): smoothing weights + normals as
    point attributes, and a mixed triangle / quad mesh with normals."""
    from conftest import GOLDEN
    stem = os.path.join(GOLDEN, f"meshio_{case}")
    for threads in (1, 3, 0):
        v, t, q, attrs = _rewrite_and_compare(ss, stem + ".ply", stem, tmp_path, threads)
    assert ("wnn" in attrs and "sw" in attrs) if case == "attr" else len(q) > 0
    # tiny chunks: hundreds of hand-overs between the formatting threads and the writing thread in every section of every format
    L = ss.load_library()
    try:
        for items, threads in ((7, 5), (1, 2), (64, 16)):
            assert L.ss_meshio_set_chunk_items(items) == 0
            _rewrite_and_compare(ss, stem + ".ply", stem, tmp_path, threads)
    finally:
        L.ss_meshio_set_chunk_items(0)
    # u32 and u64 indices, tuple input and the per-format helpers write the same bytes
    from splashsurf_b200 import io
    if case == "attr":
        io.write_vtk_mesh(str(tmp_path / "h.vtk"), v, t.astype(np.uint32), attrs)
        io.write_ply(str(tmp_path / "h.ply"), v, t.astype(np.int64), attrs)
        assert open(tmp_path / "h.vtk", "rb").read() == open(stem + ".vtk", "rb").read()
        assert open(tmp_path / "h.ply", "rb").read() == open(stem + ".ply", "rb").read()
        # the VTK reader returns what was written
        v2, t2, q2, pa, ca = io.read_vtk_mesh(stem + ".vtk")
        assert np.array_equal(v2, v) and np.array_equal(t2, t) and len(q2) == 0 and ca == {}
        assert list(pa) == list(attrs) and all(np.array_equal(pa[k], attrs[k]) for k in attrs)
        # MeshWithData.write_to_file picks the format by the extension or by name
        mwd = ss.MeshWithData(ss.TriMesh3d(v, t.astype(np.uint64)), attrs, {})
        mwd.write_to_file(str(tmp_path / "m.OBJ"))
        mwd.write_to_file(str(tmp_path / "m.dat"), file_format="obj")
        assert open(tmp_path / "m.OBJ", "rb").read() == open(tmp_path / "m.dat", "rb").read() == open(stem + ".obj", "rb").read()


def test_mesh_writers_against_live_reference_cli(ss, oracle_mod, tmp_path, reference_output):
    """Runs of the reference CLI on clouds that stress the number formatting (coordinates of 1e5 .. 1e7 and of 1e-7), an empty mesh and
    a larger mesh that spans several writer chunks (ordered hand-over between the formatting threads and the writing thread).  The
    reference's .ply of the three small cases is stored (tests/golden/reference_cli_<case>.ply.gz), its .vtk / .obj by their digests
    (tests/golden/reference_outputs.json); the larger mesh (2.3 MB) is compared where the reference (oracle/_ref) is present."""
    import gzip, subprocess, sys
    from conftest import GOLDEN, digest
    from splashsurf_b200 import io, synthetic as syn
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "import sys; sys.path.insert(0, %r); import oracle; oracle.reference().run_splashsurf(['splashsurf'] + sys.argv[1:])" % root
    p = syn.jittered_cube(5, 0.025, 2)
    big = syn.jittered_cube(14, 0.025, 4)
    cases = {"far": ((p + np.float32([123456.0, -7654321.0, 0.001])).astype(np.float32), ["-r=0.025"], []),
             "tiny": ((p * np.float32(1e-6)).astype(np.float32), ["-r=0.000000025"], []),
             "empty": (p, ["-r=0.025", "-t=50"], []),
             "big": (big, ["-r=0.025"], ["--normals=on", "--sph-normals=on"])}
    for name, (cloud, rad, flags) in cases.items():
        xyz = str(tmp_path / f"{name}.xyz")
        io.write_xyz(xyz, cloud)
        stem = str(tmp_path / f"ref_{name}")
        stored = os.path.join(GOLDEN, f"reference_cli_{name}.ply.gz")

        def run_reference():
            for ext in ("ply", "vtk", "obj"):
                subprocess.check_call([sys.executable, "-c", code, "reconstruct", xyz, *rad, "-l=2.0", "-c=0.35" if name == "big" else "-c=0.75", *flags,
                                       "-n=1", "-o", f"{stem}.{ext}", "-q"])        # one thread: the vertex order of the reference mesh is then the same in every run
            if name != "big":
                with open(f"{stem}.ply", "rb") as f, gzip.GzipFile(stored, "wb", mtime=0) as g:
                    g.write(f.read())
            return {ext: digest(open(f"{stem}.{ext}", "rb").read()) for ext in ("ply", "vtk", "obj")}
        if name == "big":
            if not oracle_mod.reference_available():
                continue
            want = run_reference()
        else:
            want = reference_output(f"mesh_writers.{name}", run_reference)
            with gzip.open(stored) as f, open(f"{stem}.ply", "wb") as g:
                g.write(f.read())
        v, t, q, attrs = _rewrite_and_compare(ss, stem + ".ply", stem, tmp_path, 4, digests=want)
        assert (len(v) == 0) == (name == "empty")
        if name == "big":
            assert len(v) > (1 << 15) and "normals" in attrs            # more than one OBJ chunk per section


def test_obj_number_formatting_is_shortest_round_trip_without_exponent(ss):
    """Rust's `{}` for f32 (obj_format.rs:33): shortest digits that read back as the same f32, positional, no trailing ".0"."""
    import ctypes as C
    L = ss.load_library()
    buf = C.create_string_buffer(80)

    def fmt(x):
        assert L.ss_format_f32(C.c_float(float(x)), buf, 80) == 0
        return buf.value.decode()
    known = [(0.0, "0"), (-0.0, "-0"), (1.0, "1"), (-2.5, "-2.5"), (16777216.0, "16777216"), (1e-7, "0.0000001"), (0.1, "0.1"),
             (1e20, "100000000000000000000"), (float("inf"), "inf"), (float("-inf"), "-inf"), (float("nan"), "NaN"),
             (3.4028235e38, "340282350000000000000000000000000000000"), (1e-45, "0.000000000000000000000000000000000000000000001"),
             (123455.984, "123455.984"), (-7654321.0, "-7654321"),
             (4.97265625, "4.9726563"), (176.390625, "176.39063"), (-1.75390625, "-1.7539063")]      # ties: Rust rounds up, Ryu to even
    for x, s in known:
        assert fmt(np.float32(x)) == s, (x, fmt(np.float32(x)), s)
    rng = np.random.default_rng(5)
    vals = rng.integers(0, 2**32, size=20000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    for x in vals:
        s = fmt(x)
        if np.isnan(x):
            assert s == "NaN"
            continue
        if np.isinf(x):
            continue
        assert "e" not in s and np.float32(s).view(np.uint32) == x.view(np.uint32)
        ref = np.format_float_positional(x, unique=True, trim="-")         # numpy rounds ties to even: same length, last digit may be one lower
        assert s == ref or (len(s) == len(ref) and s[:-1] == ref[:-1] and int(s[-1]) == int(ref[-1]) + 1)
    assert L.ss_format_f32(C.c_float(1.5), buf, 2) != 0                  # capacity too small


def test_mesh_writer_errors(ss, tmp_path):
    """write_mesh's error behaviour (io.rs:296-312): unsupported / missing extension; file that cannot be opened; attribute checks."""
    v = np.zeros((3, 3), np.float32)
    t = np.array([[0, 1, 2]], np.uint32)
    with pytest.raises(ss.SplashsurfError) as e:
        ss.write_mesh(str(tmp_path / "m.stl"), (v, t))
    assert e.value.code == ss.SS_ERR_INVALID_PARAMETER and 'Unsupported file format extension "stl"' in e.value.message
    with pytest.raises(ss.SplashsurfError) as e:
        ss.write_mesh(str(tmp_path / "mesh"), (v, t))
    assert "Unable to detect file format of mesh output file" in e.value.message
    with pytest.raises(ss.SplashsurfError) as e:
        ss.write_mesh(str(tmp_path / "no_such_dir" / "m.obj"), (v, t))
    assert e.value.code == ss.SS_ERR_IO
    with pytest.raises(ValueError):
        ss.write_mesh(str(tmp_path / "m.obj"), (v, t), point_attributes={"a": np.zeros(2, np.float32)})
    with pytest.raises(ValueError):
        ss.write_mesh(str(tmp_path / "m.obj"), (v, np.array([[0, 1, 3]], np.uint32)))
    with pytest.raises(ValueError):
        ss.write_mesh(str(tmp_path / "m.obj"), (v, t), file_format="stl")
    # u64 attributes: `uint` in a PLY (values above u32 are refused like the reference's `expect`), unsigned_long in a VTK
    from splashsurf_b200 import io
    ss.write_mesh(str(tmp_path / "u.ply"), (v, t), point_attributes={"id": np.array([1, 2, 3], np.uint64)}, cell_attributes={"c": np.ones(1, np.float32)})
    assert np.array_equal(io.read_ply_mesh(str(tmp_path / "u.ply"))[3]["id"], [1, 2, 3])
    with pytest.raises(ss.SplashsurfError) as e:
        ss.write_mesh(str(tmp_path / "u.ply"), (v, t), point_attributes={"id": np.array([1, 2, 1 << 40], np.uint64)})
    assert e.value.code == ss.SS_ERR_INDEX_TOO_SMALL
    ss.write_mesh(str(tmp_path / "u.vtk"), (v, t), point_attributes={"id": np.array([1, 2, 1 << 40], np.uint64)}, cell_attributes={"c": np.ones(1, np.float32)})
    _, _, _, pa, ca = io.read_vtk_mesh(str(tmp_path / "u.vtk"))
    assert np.array_equal(pa["id"], [1, 2, 1 << 40]) and np.array_equal(ca["c"], [1.0])


def test_obj_numbers_against_the_reference_writer_on_arbitrary_values(ss, tmp_path, reference_output):
    """`splashsurf convert --mesh in.ply -o out.obj` pushes arbitrary vertex values through the reference's OBJ writer: random bit patterns,
    subnormals, huge values, big integers and dyadic fractions -- the last two hit the exact ties where Rust rounds up and Ryu (std::to_chars)
    rounds to even, e.g. 4.97265625 -> "4.9726563".  The reference's files are pinned by their digests (tests/golden/reference_outputs.json)."""
    import subprocess, sys
    from conftest import digest
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "import sys; sys.path.insert(0, %r); import oracle; oracle.reference().run_splashsurf(['splashsurf'] + sys.argv[1:])" % root

    def ref_convert(src, out):
        subprocess.check_call([sys.executable, "-c", code, "convert", "--mesh", src, "-o", out, "--overwrite", "-q"])
        return digest(open(out, "rb").read())
    rng = np.random.default_rng(3)
    n = 30000
    parts = [rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.uint32),
             rng.integers(1, 0x00800000, size=n, dtype=np.uint64).astype(np.uint32),
             (rng.integers(1, 1 << 14, size=n) / np.exp2(rng.integers(0, 20, size=n))).astype(np.float32).view(np.uint32),
             rng.integers(1 << 24, 1 << 40, size=n).astype(np.float32).view(np.uint32),
             (-(rng.integers(1, 1 << 24, size=n).astype(np.float64) * np.exp2(-rng.integers(20, 60, size=n)))).astype(np.float32).view(np.uint32),
             np.array([4.97265625, 176.390625, 0.5, 1.5, 2.5, 8388608.5, 33554436.0, 1.7539062], np.float32).view(np.uint32)]
    bits = np.concatenate(parts)
    bits = np.concatenate([bits, np.zeros((-len(bits)) % 3, np.uint32)])
    v = bits.view(np.float32).reshape(-1, 3).copy()
    v[~np.isfinite(v)] = 1.0                                              # the reference's PLY reader is not asked to carry NaN / inf
    tri = np.array([[0, 1, 2]], np.uint32)
    ss.write_mesh(str(tmp_path / "in.ply"), (v, tri))
    want = reference_output("obj_numbers.ref.obj", lambda: ref_convert(str(tmp_path / "in.ply"), str(tmp_path / "ref.obj")))
    ss.write_mesh(str(tmp_path / "our.obj"), (v, tri), threads=3)
    assert digest(open(tmp_path / "our.obj", "rb").read()) == want
    # interoperability: the reference's own readers take this package's .ply and .vtk files, and what it writes back is what we write
    rng = np.random.default_rng(4)
    mv = rng.normal(size=(200, 3)).astype(np.float32)
    mt = rng.integers(0, 200, size=(300, 3)).astype(np.uint32)
    ss.write_mesh(str(tmp_path / "m.vtk"), (mv, mt), point_attributes={"w": rng.random(200).astype(np.float32)})
    ss.write_mesh(str(tmp_path / "m.ply"), (mv, mt))
    for src, ext in (("m.vtk", "vtk"), ("m.vtk", "obj"), ("m.ply", "vtk")):
        out = str(tmp_path / f"conv_{src[2:]}.{ext}")
        want = reference_output(f"obj_numbers.conv_{src[2:]}.{ext}", lambda: ref_convert(str(tmp_path / src), out))
        ss.write_mesh(str(tmp_path / f"mine.{ext}"), (mv, mt))                # (convert drops attributes)
        assert digest(open(tmp_path / f"mine.{ext}", "rb").read()) == want, (src, ext)


def test_vtk_point_data_reader(ss, tmp_path):
    """POINT_DATA of legacy binary VTK files: SCALARS (+ lookup table), VECTORS and FIELD arrays as SPlisHSPlasH writes them; the attribute
    loader converts like vtk_format.rs:318-346 (u32 / f32 / f64 scalars, f32 / f64 vectors -> f32) and refuses the rest."""
    from splashsurf_b200 import io
    n = 5
    pts = np.arange(3 * n, dtype=">f4")
    ids = (np.arange(n) + 7).astype(">u4")
    vel = (np.arange(3 * n) * 0.5).astype(">f4")
    dens = np.linspace(1, 2, n).astype(">f8")
    tens = np.zeros(9 * n, ">f4")
    path = str(tmp_path / "p.vtk")
    with open(path, "wb") as f:
        f.write(b"# vtk DataFile Version 4.1\nSPlisHSPlasH particle data\nBINARY\nDATASET UNSTRUCTURED_GRID\n")
        f.write(b"POINTS %d float\n" % n + pts.tobytes() + b"\n")
        f.write(b"CELLS %d %d\n" % (n, 2 * n) + np.stack([np.ones(n), np.arange(n)], 1).astype(">i4").tobytes() + b"\n")
        f.write(b"CELL_TYPES %d\n" % n + np.ones(n, ">i4").tobytes() + b"\n")
        f.write(b"POINT_DATA %d\n" % n)
        f.write(b"SCALARS id unsigned_int 1\nLOOKUP_TABLE id_table\n" + ids.tobytes() + b"\n")
        f.write(b"VECTORS force float\n" + vel.tobytes() + b"\n")
        f.write(b"FIELD FieldData 3\nvelocity 3 %d float\n" % n + vel.tobytes() + b"\ndensity 1 %d double\n" % n + dens.tobytes() +
                b"\nstress 9 %d float\n" % n + tens.tobytes() + b"\n")
    assert np.array_equal(io.read_particles(path), pts.astype("<f4").reshape(n, 3))
    d = io.read_vtk_point_data(path)
    assert list(d) == ["id", "force", "velocity", "density", "stress"] and d["id"].dtype == np.uint32 and d["density"].dtype == np.float64
    assert np.array_equal(d["id"], ids) and np.array_equal(d["velocity"], vel.reshape(n, 3)) and d["stress"].shape == (n, 9)
    a = io.read_particle_attributes(path, ["velocity", "id", "density"])
    assert all(v.dtype == np.float32 for v in a.values()) and a["velocity"].shape == (n, 3) and np.array_equal(a["id"], ids.astype(np.float32))
    with pytest.raises(ValueError, match='Missing attribute\\(s\\) "pressure" in input file'):
        io.read_particle_attributes(path, ["pressure"])
    with pytest.raises(ValueError, match="Unsupported number of components"):
        io.read_particle_attributes(path, ["stress"])
    assert io.read_particle_attributes(path, []) == {}
    # files of this package's own writer carry their attributes as SCALARS
    ss.write_mesh(str(tmp_path / "m.vtk"), (pts.astype("<f4").reshape(n, 3), np.array([[0, 1, 2]], np.uint32)),
                  point_attributes={"w": np.ones(n, np.float32), "nrm": np.ones((n, 3), np.float32)})
    d = io.read_vtk_point_data(str(tmp_path / "m.vtk"))
    assert d["w"].shape == (n,) and d["nrm"].shape == (n, 3)
