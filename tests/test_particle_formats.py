"""Particle file formats either side of the hot path (SURVEY.md 8f #3; splashsurf_lib/src/io.rs:17-43, splashsurf/src/io.rs:195-235):
every format the reference reads (.vtk legacy ASCII / BINARY, .vtu XML in its encodings, .ply, .bgeo, .json, .xyz) and writes
(.vtk, .bgeo, .json), the attribute inputs of `-a`, and the `convert` subcommand -- self-contained round trips plus comparisons with the
reference CLI (its outputs stored in tests/golden/reference_outputs.json) and the reference's data files (tests/golden/reference_data)."""
import base64
import gzip
import os
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

from splashsurf_b200 import io, particle_formats as pf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_CODE = "import sys; sys.path.insert(0, %r); import oracle; oracle.reference().run_splashsurf(['splashsurf'] + sys.argv[1:])" % ROOT


def _cloud(n=257, seed=3):
    rng = np.random.default_rng(seed)
    p = rng.uniform(-2.0, 3.0, size=(n, 3)).astype(np.float32)
    # values that stress the number formatting: tiny, huge, exact integers, negative zero
    p[:6] = np.float32([[0.1, 0.2, 0.3], [1.0, 2.0, 3.0], [-1e-7, 1e16, 5e-5], [123456.789, 0.5, 1e-5], [-0.0, 1e-30, 3e38], [16777216.0, 1e15, 1e17]])
    return p


def _ref(*args):
    return subprocess.run([sys.executable, "-c", REF_CODE, *args, "-q"], capture_output=True, text=True)


def _file_digest(path):
    """Digest of a written file; a .bgeo is compared by its gzip header and its uncompressed contents."""
    from conftest import digest
    b = open(path, "rb").read()
    return digest(b[:10], gzip.decompress(b)) if path.endswith(".bgeo") else digest(b)


def _ref_file_digest(*args):
    """Runs the reference CLI with `args` (the output file follows "-o") and returns the digest of the file it wrote."""
    r = _ref(*args)
    assert r.returncode == 0, r.stderr[-600:]
    return _file_digest(args[list(args).index("-o") + 1])


# ---------------------------------------------------------------------------------------------------- test-side file writers
def _vtu(path, points, point_data, *, mode, compressed=False, header="UInt64", byte_order="LittleEndian", appended_encoding="raw",
         split_b64=True, kind="UnstructuredGrid"):
    """A VTU / VTP writer covering the encodings VTK itself produces: mode = ascii | binary | appended."""
    bo = "<" if byte_order == "LittleEndian" else ">"
    hd = bo + ("u8" if header == "UInt64" else "u4")
    names = {"f4": "Float32", "f8": "Float64", "i8": "Int64", "u4": "UInt32", "u1": "UInt8", "i4": "Int32"}

    def block(a):
        raw = a.astype(bo + a.dtype.str[1:]).tobytes()
        if not compressed:
            return np.array([len(raw)], hd).tobytes(), raw
        bs = 1 << 10                                                       # small blocks: several per array
        chunks = [raw[i:i + bs] for i in range(0, len(raw), bs)] or []
        comp = [zlib.compress(c) for c in chunks]
        last = len(chunks[-1]) % bs if chunks else 0
        h = np.array([len(chunks), bs, last] + [len(c) for c in comp], hd).tobytes()
        return h, b"".join(comp)
    appended = []

    def data_array(a, name, comps):
        t = names[a.dtype.str[1:]]
        attr = f'type="{t}" Name="{name}" NumberOfComponents="{comps}"'
        if mode == "ascii":
            return f'<DataArray {attr} format="ascii">\n{" ".join(repr(v) for v in a.reshape(-1).tolist())}\n</DataArray>'
        h, d = block(a.reshape(-1))
        if mode == "binary":
            txt = (base64.b64encode(h) + base64.b64encode(d)) if (split_b64 or compressed) else base64.b64encode(h + d)
            return f'<DataArray {attr} format="binary">\n{txt.decode()}\n</DataArray>'
        if appended_encoding == "raw":
            off = sum(len(x) for x in appended)
            appended.append(h + d)
        else:
            off = sum(len(x) for x in appended)
            appended.append((base64.b64encode(h) + base64.b64encode(d)) if (split_b64 or compressed) else base64.b64encode(h + d))
        return f'<DataArray {attr} format="appended" offset="{off}"/>'
    n = len(points)
    xml = ['<?xml version="1.0"?>', f'<VTKFile type="{kind}" version="1.0" byte_order="{byte_order}" header_type="{header}"'
           + (' compressor="vtkZLibDataCompressor"' if compressed else "") + ">", f"<{kind}>",
           f'<Piece NumberOfPoints="{n}" ' + (f'NumberOfCells="{n}"' if kind == "UnstructuredGrid" else f'NumberOfVerts="{n}"') + ">", "<PointData>"]
    for name, a in point_data.items():
        xml.append(data_array(a, name, 1 if a.ndim == 1 else a.shape[1]))
    xml += ["</PointData>", "<Points>", data_array(points, "Points", 3), "</Points>"]
    conn, offs = np.arange(n, dtype=np.int64), np.arange(1, n + 1, dtype=np.int64)
    if kind == "UnstructuredGrid":
        xml += ["<Cells>", data_array(conn, "connectivity", 1), data_array(offs, "offsets", 1), data_array(np.ones(n, np.uint8), "types", 1), "</Cells>"]
    else:
        xml += ["<Verts>", data_array(conn, "connectivity", 1), data_array(offs, "offsets", 1), "</Verts>"]
    xml += ["</Piece>", f"</{kind}>"]
    body = "\n".join(xml).encode()
    if mode == "appended":
        body += f'\n<AppendedData encoding="{appended_encoding}">\n_'.encode() + b"".join(appended) + b"\n</AppendedData>"
    body += b"\n</VTKFile>\n"
    open(path, "wb").write(body)


def _legacy_vtk(path, points, point_data, *, binary, typ="float"):
    dt = ">f4" if typ == "float" else ">f8"
    n = len(points)
    with open(path, "wb") as f:
        f.write(b"# vtk DataFile Version 4.2\nsome particles\n" + (b"BINARY" if binary else b"ASCII") + b"\nDATASET UNSTRUCTURED_GRID\n")
        f.write(f"POINTS {n} {typ}\n".encode())

        def arr(a, d):
            if binary:
                f.write(a.astype(d).tobytes() + b"\n")
            else:
                f.write((" ".join(repr(v) for v in a.reshape(-1).tolist()) + "\n").encode())
        arr(points, dt)
        cells = np.stack([np.ones(n, np.int32), np.arange(n, dtype=np.int32)], axis=1)
        f.write(f"CELLS {n} {2 * n}\n".encode())
        arr(cells, ">i4")
        f.write(f"CELL_TYPES {n}\n".encode())
        arr(np.ones(n, np.int32), ">i4")
        f.write(f"POINT_DATA {n}\n".encode())
        for name, a in point_data.items():
            t = {"f4": "float", "f8": "double", "u4": "unsigned_int", "i8": "long"}[a.dtype.str[1:]]
            if a.ndim == 1:
                f.write(f"SCALARS {name} {t} 1\nLOOKUP_TABLE default\n".encode())
            else:
                f.write(f"VECTORS {name} {t}\n".encode())
            arr(a, ">" + a.dtype.str[1:])


def _ply_particles(path, points, *, fmt, extra=True):
    n = len(points)
    head = f"ply\nformat {fmt} 1.0\ncomment made by a test\nelement vertex {n}\nproperty float x\nproperty float y\nproperty float z\n"
    if extra:
        head += "property uchar red\nproperty double weight\n"
    head += "end_header\n"
    with open(path, "wb") as f:
        f.write(head.encode())
        if fmt == "ascii":
            for i, q in enumerate(points.tolist()):
                f.write((" ".join(repr(v) for v in q) + (f" {i % 256} {i * 0.5!r}" if extra else "") + "\n").encode())
        else:
            bo = "<" if fmt == "binary_little_endian" else ">"
            dt = [("x", bo + "f4"), ("y", bo + "f4"), ("z", bo + "f4")] + ([("red", "u1"), ("weight", bo + "f8")] if extra else [])
            rec = np.zeros(n, dtype=dt)
            rec["x"], rec["y"], rec["z"] = points[:, 0], points[:, 1], points[:, 2]
            if extra:
                rec["red"] = np.arange(n) % 256
                rec["weight"] = np.arange(n) * 0.5
            f.write(rec.tobytes())


def _bgeo_with_attributes(path, points, attrs, *, compress):
    """attrs: ordered name -> int32 (n,) | float32 (n,) | float32 (n, k)."""
    n = len(points)
    out = b"Bgeo" + struct.pack(">Bi8i", 86, 5, n, 0, 0, 0, len(attrs), 0, 0, 0)
    fields = [("p", ">f4", (3,)), ("w", ">f4")]
    for name, a in attrs.items():
        size = 1 if a.ndim == 1 else a.shape[1]
        typ = 1 if a.dtype.kind == "i" else (0 if a.ndim == 1 else 5)
        out += struct.pack(">H", len(name)) + name.encode() + struct.pack(">Hi", size, typ) + struct.pack(f">{size}i", *([0] * size))
        fields.append((name, ">i4" if typ == 1 else ">f4", (size,)) if a.ndim > 1 else (name, ">i4" if typ == 1 else ">f4"))
    rec = np.zeros(n, dtype=fields)
    rec["p"], rec["w"] = points, 1.0
    for name, a in attrs.items():
        rec[name] = a
    out += rec.tobytes() + b"\x00\xff"
    open(path, "wb").write(gzip.compress(out) if compress else out)


# ------------------------------------------------------------------------------------------------------------------- tests
def test_json_numbers_follow_ryu():
    """serde_json prints f64 through Ryu: shortest digits, positional for -5 < e10 <= 16 (json_format.rs:55-94)."""
    known = [(0.0, "0.0"), (-0.0, "-0.0"), (1.0, "1.0"), (0.5, "0.5"), (1e16, "1e16"), (1e15, "1000000000000000.0"), (1.5e16, "1.5e16"),
             (123456.7890625, "123456.7890625"), (1e-5, "0.00001"), (1e-6, "1e-6"), (9.999999747378752e-6, "9.999999747378752e-6"),
             (0.00004999999873689376, "0.00004999999873689376"), (-1.0000000116860974e-7, "-1.0000000116860974e-7"),
             (1.0000000272564224e16, "1.0000000272564224e16"), (float(np.float32(0.1)), "0.10000000149011612"), (5e-324, "5e-324"),
             (1.7976931348623157e308, "1.7976931348623157e308"), (123.0, "123.0"), (1234567890123456.0, "1234567890123456.0"),
             (12345678901234567.0, "1.2345678901234568e16"), (float("nan"), "null"), (float("inf"), "null")]
    for x, s in known:
        assert pf.format_f64_json(x) == s, (x, pf.format_f64_json(x), s)
    rng = np.random.default_rng(0)
    for x in rng.integers(0, 2**32, size=5000, dtype=np.uint64).astype(np.uint32).view(np.float32):
        if np.isfinite(x):
            assert float(pf.format_f64_json(float(x))) == float(x)


def test_round_trips_of_every_writer(tmp_path):
    p = _cloud()
    for name, kw in (("a.vtk", {}), ("a.bgeo", {}), ("b.bgeo", {"enable_compression": False}), ("a.json", {})):
        path = str(tmp_path / name)
        pf.write_particle_positions(path, p, **kw)
        assert np.array_equal(pf.particles_from_file(path).view(np.uint32), p.view(np.uint32)), name
    raw = open(tmp_path / "b.bgeo", "rb").read()
    assert raw[:4] == b"Bgeo" and raw[-2:] == b"\x00\xff" and len(raw) == 41 + 16 * len(p) + 2
    gz = open(tmp_path / "a.bgeo", "rb").read()
    assert gz[:10] == b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x04\xff" and gzip.decompress(gz) == raw          # flate2's header, same payload
    io.write_particles(str(tmp_path / "a.xyz"), p)
    assert np.array_equal(io.read_particles(str(tmp_path / "a.xyz")), p)
    # upper-case extensions are recognised like in the reference (to_lowercase)
    pf.write_particle_positions(str(tmp_path / "C.JSON"), p[:3])
    assert np.array_equal(pf.particles_from_file(str(tmp_path / "C.JSON")), p[:3])
    with pytest.raises(ValueError, match="Unsupported file format extension"):
        pf.write_particle_positions(str(tmp_path / "a.xyz2"), p)
    with pytest.raises(ValueError, match="Unable to detect file format"):
        pf.particles_from_file(str(tmp_path / "noext"))
    # empty clouds
    for name in ("e.vtk", "e.bgeo", "e.json"):
        pf.write_particle_positions(str(tmp_path / name), np.zeros((0, 3), np.float32))
        assert pf.particles_from_file(str(tmp_path / name)).shape == (0, 3)


VTU_VARIANTS = [dict(mode="ascii"), dict(mode="binary"), dict(mode="binary", split_b64=False), dict(mode="binary", compressed=True),
                dict(mode="binary", header="UInt32"), dict(mode="appended"), dict(mode="appended", compressed=True),
                dict(mode="appended", appended_encoding="base64"), dict(mode="appended", appended_encoding="base64", split_b64=False),
                dict(mode="appended", appended_encoding="base64", compressed=True), dict(mode="appended", byte_order="BigEndian", header="UInt32"),
                dict(mode="appended", compressed=True, kind="PolyData"), dict(mode="ascii", kind="PolyData")]


def _point_data(n, seed=5):
    rng = np.random.default_rng(seed)
    return {"velocity": rng.normal(size=(n, 3)), "density": rng.uniform(900, 1100, n).astype(np.float32), "id": np.arange(n, dtype=np.uint32),
            "index": np.arange(n, dtype=np.int64), "pressure": rng.uniform(0, 1e5, n)}


@pytest.mark.parametrize("variant", VTU_VARIANTS, ids=lambda v: "-".join(f"{k}={x}" for k, x in v.items()))
def test_vtu_encodings(tmp_path, variant):
    n = 333                                                                # > one 1 KiB compression block per array
    p64 = _cloud(n).astype(np.float64) + 1e-9
    data = _point_data(n)
    path = str(tmp_path / "c.vtu")
    _vtu(path, p64, data, **variant)
    assert np.array_equal(pf.particles_from_file(path), p64.astype(np.float32))
    pts, pd = pf.read_vtk(path)
    assert pts.dtype == np.float64 and np.array_equal(pts, p64)
    assert list(pd.keys()) == list(data) and all(np.array_equal(pd[k], data[k]) and pd[k].dtype == data[k].dtype for k in data)
    a = pf.particle_attributes_from_file(path, ["density", "velocity", "id", "pressure"])
    assert list(a) == ["density", "velocity", "id", "pressure"] and all(v.dtype == np.float32 for v in a.values())
    assert np.array_equal(a["velocity"], data["velocity"].astype(np.float32)) and np.array_equal(a["id"], data["id"].astype(np.float32))
    with pytest.raises(ValueError, match="Unsupported IOBuffer scalar data type"):
        pf.particle_attributes_from_file(path, ["index"])                  # i64 scalars: vtk_format.rs:318-333
    with pytest.raises(ValueError, match='Missing attribute\\(s\\) "nope"'):
        pf.particle_attributes_from_file(path, ["density", "nope"])


@pytest.mark.parametrize("binary", [True, False])
@pytest.mark.parametrize("typ", ["float", "double"])
def test_legacy_vtk_ascii_binary_float_double(tmp_path, binary, typ):
    n = 100
    p = _cloud(n)
    pts = p if typ == "float" else p.astype(np.float64) + 1e-9
    data = {"velocity": np.random.default_rng(1).normal(size=(n, 3)).astype(np.float32), "density": np.linspace(900, 1100, n),
            "id": np.arange(n, dtype=np.uint32), "index": np.arange(n, dtype=np.int64)}
    path = str(tmp_path / "c.vtk")
    _legacy_vtk(path, pts, data, binary=binary, typ=typ)
    assert np.array_equal(pf.particles_from_file(path), pts.astype(np.float32))
    assert np.array_equal(io.read_vtk_points(path), pts.astype(np.float32))
    a = io.read_particle_attributes(path, ["id", "velocity", "density"])
    assert np.array_equal(a["id"], data["id"].astype(np.float32)) and np.array_equal(a["velocity"], data["velocity"])
    assert np.array_equal(a["density"], data["density"].astype(np.float32))
    with pytest.raises(ValueError, match="Unsupported IOBuffer scalar data type"):
        io.read_particle_attributes(path, ["index"])


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
def test_ply_particles(tmp_path, fmt):
    p = _cloud(90)
    path = str(tmp_path / "c.ply")
    for extra in (False, True):
        _ply_particles(path, p, fmt=fmt, extra=extra)
        assert np.array_equal(pf.particles_from_file(path), p)
    # double coordinates are refused like in the reference (ply_format.rs:55-62)
    if fmt == "ascii":
        b = open(path, "rb").read().replace(b"property float x", b"property double x")
        open(path, "wb").write(b)
        with pytest.raises(ValueError, match="expected float"):
            pf.particles_from_file(path)


def test_bgeo_attributes_and_errors(tmp_path):
    n = 64
    p = _cloud(n)
    rng = np.random.default_rng(2)
    attrs = {"velocity": rng.normal(size=(n, 3)).astype(np.float32), "density": rng.uniform(900, 1100, n).astype(np.float32),
             "id": np.arange(n, dtype=np.int32), "uv": rng.normal(size=(n, 2)).astype(np.float32)}
    for compress in (False, True):
        path = str(tmp_path / f"c{int(compress)}.bgeo")
        _bgeo_with_attributes(path, p, attrs, compress=compress)
        q, a = pf.read_bgeo(path)
        assert np.array_equal(q, p) and list(a) == list(attrs) and all(np.array_equal(a[k], attrs[k]) for k in attrs)
        got = pf.particle_attributes_from_file(path, ["density", "velocity", "id"])
        assert got["id"].dtype == np.uint64 and np.array_equal(got["id"], np.arange(n)) and np.array_equal(got["velocity"], attrs["velocity"])
        with pytest.raises(ValueError, match="unsupported vector attribute size: 2"):
            pf.particle_attributes_from_file(path, ["uv"])
        with pytest.raises(ValueError, match='Missing attribute\\(s\\) "rho"'):
            pf.particle_attributes_from_file(path, ["rho"])
    raw = open(tmp_path / "c0.bgeo", "rb").read()
    for bad, msg in ((b"Hgeo" + raw[4:], "MagicBytesNotFound"), (b"\x7fNSJ" + raw[4:], "UnsupportedFormatVersion"),
                     (raw[:5] + struct.pack(">i", 4) + raw[9:], "UnsupportedFormatVersion"), (raw[:100], "unexpected end of file")):
        open(tmp_path / "bad.bgeo", "wb").write(bad)
        with pytest.raises(ValueError, match=msg):
            pf.read_bgeo(str(tmp_path / "bad.bgeo"))
    # string attributes are refused (bgeo_format.rs:448-452)
    _bgeo_with_attributes(str(tmp_path / "s.bgeo"), p, {"id": np.arange(n, dtype=np.int32)}, compress=False)
    b = bytearray(open(tmp_path / "s.bgeo", "rb").read())
    b[41 + 2 + 2 + 2:41 + 2 + 2 + 2 + 4] = struct.pack(">i", 4)
    open(tmp_path / "s.bgeo", "wb").write(bytes(b))
    with pytest.raises(ValueError, match="UnsupportedAttributeType\\(IndexedString\\)"):
        pf.read_bgeo(str(tmp_path / "s.bgeo"))


def test_json_reader_errors(tmp_path):
    for text, msg in (("[[1,2,3],[4,5]]", "Parsing of JSON structure"), ("{\"a\": 1}", "Parsing of JSON structure"), ("[[1,2,3", "Not a valid JSON file"),
                      ("[[1,2,\"x\"]]", "Parsing of JSON structure")):
        open(tmp_path / "b.json", "w").write(text)
        with pytest.raises(ValueError, match=msg):
            pf.read_json(str(tmp_path / "b.json"))
    open(tmp_path / "i.json", "w").write("[[1, 2, 3], [4.5, -5e-1, 6]]")
    assert np.array_equal(pf.read_json(str(tmp_path / "i.json")), np.float32([[1, 2, 3], [4.5, -0.5, 6]]))


def test_writers_and_readers_beside_the_reference_cli(tmp_path, reference_output):
    """The reference's `convert` writes .vtk / .bgeo / .json from a cloud: our writers write its bytes (digests of the reference's
    files in tests/golden/reference_outputs.json) and our readers return the particles; the files written by this test's own writers
    (VTU encodings, legacy ASCII / double, PLY flavours, BGEO with attributes) are read identically by the reference: the .json it
    converts them to is the file our writer makes of the expected particles."""
    p = _cloud(1500)
    xyz = str(tmp_path / "c.xyz")
    io.write_xyz(xyz, p)
    for ext in ("vtk", "bgeo", "json"):
        ref = str(tmp_path / f"ref.{ext}")
        want = reference_output(f"convert_particles.{ext}", lambda: _ref_file_digest("convert", "--particles", xyz, "-o", ref))
        mine = str(tmp_path / f"mine.{ext}")
        pf.write_particle_positions(mine, p)
        assert _file_digest(mine) == want, ext
        assert np.array_equal(pf.particles_from_file(mine).view(np.uint32), p.view(np.uint32)), ext
    # our files through the reference's readers
    n = 400
    q = _cloud(n, seed=9)
    q64 = q.astype(np.float64) + 1e-9
    files = []
    for i, variant in enumerate(VTU_VARIANTS):
        # vtkio 0.6.3 (the reference's reader) takes inline / appended base64 arrays only when the length prefix and the data are ONE
        # base64 block, and its XML reader trips over raw appended bytes that look like markup; VTK's own layouts (two blocks, raw
        # appended data, compression) are covered by test_vtu_encodings above
        if not (variant["mode"] == "ascii" or variant.get("split_b64") is False) or variant.get("kind") == "PolyData":
            continue
        path = str(tmp_path / f"v{i}.vtu")
        _vtu(path, q64, _point_data(n), **variant)
        files.append((path, q64.astype(np.float32)))
    for binary in (True, False):
        for typ in ("float", "double"):
            path = str(tmp_path / f"l{int(binary)}{typ}.vtk")
            _legacy_vtk(path, q if typ == "float" else q64, {"density": np.linspace(0, 1, n).astype(np.float32)}, binary=binary, typ=typ)
            files.append((path, (q if typ == "float" else q64).astype(np.float32)))
    for fmt in ("ascii", "binary_little_endian", "binary_big_endian"):
        path = str(tmp_path / f"p_{fmt}.ply")
        _ply_particles(path, q, fmt=fmt)
        files.append((path, q))
    path = str(tmp_path / "attr.bgeo")
    _bgeo_with_attributes(path, q, {"velocity": np.ones((n, 3), np.float32), "id": np.arange(n, dtype=np.int32)}, compress=True)
    files.append((path, q))
    for path, expect in files:
        name = os.path.basename(path)
        theirs = reference_output(f"read_by_reference.{name}", lambda: _ref_file_digest("convert", "--particles", path, "-o", path + ".json"))
        pf.write_particle_positions(path + ".expect.json", expect)
        assert _file_digest(path + ".expect.json") == theirs, name
        assert np.array_equal(pf.particles_from_file(path), expect), name


def test_convert_subcommand_beside_the_reference_cli(ss, tmp_path, reference_output):
    """`python -m splashsurf_b200 convert` against `splashsurf convert` (digests of its files in tests/golden/reference_outputs.json):
    particle conversion with the half-open domain filter, mesh conversion .vtk / .ply -> .obj / .vtk / .ply, the overwrite check."""
    from splashsurf_b200.__main__ import main
    p = _cloud(800)
    xyz = str(tmp_path / "c.xyz")
    io.write_xyz(xyz, p)
    box = ["--domain-min", "-1.0", "-0.5", "-2", "--domain-max", "2.0", "1.5", str(float(p[10, 2]))]       # a particle exactly on the open face
    for ext in ("vtk", "json", "bgeo"):
        ref, mine = str(tmp_path / f"r.{ext}"), str(tmp_path / f"m.{ext}")
        want = reference_output(f"convert_particles_in_box.{ext}", lambda: _ref_file_digest("convert", "--particles", xyz, "-o", ref, *box))
        assert main(["convert", "--particles", xyz, "-o", mine, *box]) == 0
        assert _file_digest(mine) == want, ext
    kept = pf.particles_from_file(str(tmp_path / "m.json"))
    assert 0 < len(kept) < len(p) and np.all(kept[:, 2] < p[10, 2])
    assert main(["convert", "--particles", xyz, "-o", str(tmp_path / "m.json")]) == 1                       # exists, no --overwrite
    assert main(["convert", "--particles", xyz, "-o", str(tmp_path / "m.json"), "--overwrite"]) == 0
    assert main(["convert", "-o", str(tmp_path / "x.json")]) == 1
    assert main(["convert", "--particles", xyz, "-o", str(tmp_path / "x.obj")]) == 1
    # meshes: the committed reference files of the mesh writers as inputs
    g = os.path.join(ROOT, "tests", "golden")
    for src in ("meshio_attr.vtk", "meshio_attr.ply"):
        for ext in ("obj", "vtk", "ply"):
            ref, mine = str(tmp_path / f"r_{src}.{ext}"), str(tmp_path / f"m_{src}.{ext}")
            want = reference_output(f"convert_mesh.{src}.{ext}", lambda: _ref_file_digest("convert", "--mesh", os.path.join(g, src), "-o", ref))
            assert main(["convert", "--mesh", os.path.join(g, src), "-o", mine]) == 0
            assert _file_digest(mine) == want, (src, ext)
    # a mesh with quads is not a triangle mesh for either CLI
    assert reference_output("convert_mesh.meshio_quad.vtk.obj.refused",
                            lambda: _ref("convert", "--mesh", os.path.join(g, "meshio_quad.vtk"), "-o", str(tmp_path / "q.obj")).returncode != 0)
    assert main(["convert", "--mesh", os.path.join(g, "meshio_quad.vtk"), "-o", str(tmp_path / "q.obj")]) == 1


def test_reference_fixture_files_when_present(tmp_path, reference_output):
    """Every particle file of the reference's data/ directory (copies under tests/golden/reference_data): our reader returns the
    particles the reference's own reader returns -- the .json its `convert` writes of a file (stored by its digest in
    tests/golden/reference_outputs.json) is the file our writer makes of what our reader read.  Two files its reader refuses -- a
    VTK 5.1 legacy file and one VTU -- are read here as well."""
    d = os.path.join(ROOT, "tests", "golden", "reference_data")
    seen = 0
    for f in sorted(os.listdir(d)):
        ext = f.rsplit(".", 1)[-1]
        if ext not in ("vtk", "vtu", "bgeo", "ply") or f in ("cube_8_particles.vtk", "fluid_250_particles.vtu"):
            continue
        out = str(tmp_path / "o.json")
        want = reference_output(f"read_reference_data.{f}", lambda: _ref_file_digest("convert", "--particles", os.path.join(d, f), "-o", out, "--overwrite"))
        pf.write_particle_positions(str(tmp_path / "mine.json"), pf.particles_from_file(os.path.join(d, f)))
        assert _file_digest(str(tmp_path / "mine.json")) == want, f
        os.remove(tmp_path / "mine.json")
        seen += 1
    assert seen >= 15
    assert len(pf.particles_from_file(os.path.join(d, "cube_8_particles.vtk"))) == 8 and len(pf.particles_from_file(os.path.join(d, "fluid_250_particles.vtu"))) == 250


def test_reference_io_unit_tests(tmp_path):
    """The unit tests inside the reference's io modules, on its own data files (copies under tests/golden/reference_data):
    bgeo_format.rs:864-967, vtk_format.rs:406-450, ply_format.rs:274-310, obj_format.rs:168-192."""
    d = os.path.join(ROOT, "tests", "golden", "reference_data")
    # test_bgeo_read_dam_break / _attributes
    path = os.path.join(d, "dam_break_frame_9_6859_particles.bgeo")
    p, attrs = pf.read_bgeo(path)
    assert len(p) == 6859 and len(attrs) == 3
    lo, hi = p.min(axis=0), p.max(axis=0)
    assert np.all(lo >= np.float32([-2.0, 0.03, -0.8])) and np.all(hi < np.float32([-0.3, 0.7, 0.72]))
    a = pf.particle_attributes_from_file(path, ["id", "density", "velocity"])
    assert a["id"].dtype == np.uint64 and a["density"].dtype == np.float32 and a["velocity"].shape == (6859, 3)
    assert a["id"][:3].tolist() == [30, 11, 12]
    assert a["density"][:3].tolist() == [np.float32(1000.1286), np.float32(1001.53424), np.float32(1001.6626)]
    assert a["velocity"][0].tolist() == [np.float32(0.3670507), np.float32(-0.41762838), np.float32(0.42659923)]
    # test_bgeo_write_dam_break: uncompressed write, read back
    out = str(tmp_path / "w.bgeo")
    pf.write_bgeo(out, p, enable_compression=False)
    q = pf.read_bgeo(out)[0]
    assert len(q) == 6859 and np.array_equal(q.view(np.uint32), p.view(np.uint32))
    # vtk_format.rs:425-450
    for name, n in (("cube_8_particles.vtu", 8), ("cube_8_particles.vtk", 8), ("double_dam_break_frame_01_4732_particles.vtk", 4732),
                    ("fluid_encoded_250_particles.vtu", 250), ("fluid_250_particles.vtu", 250)):
        assert len(pf.particles_from_file(os.path.join(d, name))) == n, name
    # ply_format.rs:274-310
    v, t, a = pf.read_ply_surface_mesh(os.path.join(d, "cube.ply"))
    assert (len(v), len(t), list(a)) == (24, 12, [])
    v, t, a = pf.read_ply_surface_mesh(os.path.join(d, "cube_normals.ply"))
    assert (len(v), len(t)) == (24, 12) and a["normals"].shape == (24, 3)
    # obj_format.rs:168-192
    for name in ("icosphere.obj", "icosphere_normals.obj"):
        v, t = io.read_obj(os.path.join(d, name))
        assert (len(v), len(t)) == (42, 80) and int(t.max()) == 41
