"""`python -m splashsurf_b200 reconstruct <particles> -r <radius> -l <smoothing length> -c <cube size> [-o out.obj]`

and `python -m splashsurf_b200 convert (--particles <file> | --mesh <file>) -o <file> [--overwrite] [--domain-min x y z --domain-max x y z]`
(splashsurf/src/convert.rs).

A thin stand-in for `splashsurf reconstruct` (splashsurf/src/reconstruct.rs:36-380): the relative `-l` / `-c` values are multiplied
by the particle radius like the reference CLI does (reconstruct.rs:628-629); the post-processing switches (`--mesh-cleanup`,
`--decimate-barnacles`, `--mesh-smoothing-iters`, `--normals`, `--sph-normals`, `--generate-quads`, `--mesh-aabb-min/-max`,
`--check-mesh`, `-a <attribute>` from a VTK / VTU / BGEO particle file) go through `reconstruction_pipeline` with the reference's option names and defaults, and the output file (`.vtk`,
`.ply`, `.obj` with the attributes the reference writes) comes from the library's writer, byte for byte the reference CLI's file."""
import argparse
import sys
import time

import numpy as np


def convert(a) -> int:
    """`convert_subcommand` (splashsurf/src/convert.rs:58-152): particles .vtk / .vtu / .bgeo / .ply / .xyz / .json -> .vtk / .bgeo / .json
    (optionally filtered by a half-open domain box, aabb.rs:220-222), or a triangle mesh .vtk / .ply -> .obj / .vtk / .ply."""
    import os
    from . import io, particle_formats as pf
    if (a.input_particles is None) == (a.input_mesh is None):
        print("Aborting: " + ("No input file specified, either a particle or mesh input file has to be specified." if a.input_particles is None
                              else "the argument '--particles' cannot be used with '--mesh'"), file=sys.stderr)
        return 1
    if (a.domain_min is None) != (a.domain_max is None):
        print("Aborting: --domain-min and --domain-max have to be specified together", file=sys.stderr)
        return 1
    if not a.overwrite and os.path.exists(a.output_file):
        print(f'Aborting: Output file "{a.output_file}" already exists. Use overwrite flag to ignore this.', file=sys.stderr)
        return 1
    try:
        if a.input_particles is not None:
            p = pf.particles_from_file(a.input_particles)
            if a.domain_min is not None:
                lo, hi = np.asarray(a.domain_min, np.float64).astype(np.float32), np.asarray(a.domain_max, np.float64).astype(np.float32)
                p = p[np.all(p >= lo, axis=1) & np.all(p < hi, axis=1)]
            pf.write_particle_positions(a.output_file, p)
        else:
            ext = os.path.splitext(a.input_mesh)[1].lower()
            if ext == ".vtk":
                v, t = pf.read_vtk_surface_mesh(a.input_mesh)
                attrs = {}
            elif ext == ".ply":
                v, t, attrs = pf.read_ply_surface_mesh(a.input_mesh)
            elif not ext:
                raise ValueError("Unable to detect file format of mesh input file (file name has to end with supported extension)")
            else:
                raise ValueError(f'Unsupported file format extension "{ext[1:]}" for reading surface meshes')
            io.write_mesh(a.output_file, (v, t), point_attributes=attrs or None)
    except (ValueError, OSError) as e:
        print(f"Error occurred: {e}", file=sys.stderr)
        return 1
    return 0


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m splashsurf_b200")
    sub = ap.add_subparsers(dest="cmd", required=True)
    r = sub.add_parser("reconstruct")
    r.add_argument("input")
    r.add_argument("-r", "--particle-radius", type=float, required=True)
    r.add_argument("-l", "--smoothing-length", type=float, required=True)
    r.add_argument("-c", "--cube-size", type=float, required=True)
    r.add_argument("-t", "--surface-threshold", type=float, default=0.6)
    r.add_argument("--rest-density", type=float, default=1000.0)
    r.add_argument("--subdomain-cubes", type=int, default=64)
    r.add_argument("--subdomain-grid", choices=["on", "off"], default="on")
    r.add_argument("--simd", choices=["on", "off"], default="on")
    r.add_argument("--sph-normals", choices=["on", "off"], default="off")
    r.add_argument("-a", "--interpolate_attribute", dest="interpolate_attributes", action="append", default=[], metavar="ATTRIBUTE_NAME")
    # post-processing, names and defaults of the reference CLI (reconstruct.rs:150-300)
    r.add_argument("--normals", choices=["on", "off"], default="off")
    r.add_argument("--normals-smoothing-iters", type=int, default=None)
    r.add_argument("--mesh-cleanup", choices=["on", "off"], default=None)        # on by default when smoothing runs (reconstruct.rs:200-213)
    r.add_argument("--mesh-cleanup-snap-dist", type=float, default=None)
    r.add_argument("--decimate-barnacles", choices=["on", "off"], default="off")
    r.add_argument("--keep-verts", choices=["on", "off"], default="off")
    r.add_argument("--mesh-smoothing-iters", type=int, default=None)
    r.add_argument("--mesh-smoothing-weights", choices=["on", "off"], default="off")
    r.add_argument("--mesh-smoothing-weights-normalization", type=float, default=13.0)
    r.add_argument("--output-smoothing-weights", choices=["on", "off"], default="off")
    r.add_argument("--output-raw-normals", choices=["on", "off"], default="off")
    r.add_argument("--generate-quads", choices=["on", "off"], default="off")
    r.add_argument("--quad-max-edge-diag-ratio", type=float, default=1.75)
    r.add_argument("--quad-max-normal-angle", type=float, default=10.0)
    r.add_argument("--quad-max-interior-angle", type=float, default=135.0)
    r.add_argument("--mesh-aabb-min", type=float, nargs=3, default=None)
    r.add_argument("--mesh-aabb-max", type=float, nargs=3, default=None)
    r.add_argument("--mesh-aabb-clamp-verts", choices=["on", "off"], default="off")
    r.add_argument("--check-mesh", choices=["on", "off"], default="off")
    r.add_argument("-o", "--output-file", default=None)
    r.add_argument("--output-dir", default=None)
    r.add_argument("-s", "--start-index", type=int, default=None)
    r.add_argument("-e", "--end-index", type=int, default=None)
    r.add_argument("-d", "--double-precision", choices=["on", "off"], default="off")
    r.add_argument("--particle-aabb-min", type=float, nargs=3, default=None)
    r.add_argument("--particle-aabb-max", type=float, nargs=3, default=None)
    r.add_argument("--mt-files", choices=["on", "off"], default="off")              # accepted: frames are sharded over GPUs instead (--shard / launcher)
    r.add_argument("--mt-particles", choices=["on", "off"], default="on")
    r.add_argument("-n", "--num-threads", type=int, default=None)                    # accepted, no meaning on the device
    r.add_argument("--subdomain-grid-auto-disable", choices=["on", "off"], default="on")
    r.add_argument("--output-raw-mesh", choices=["on", "off"], default="off")
    r.add_argument("--check-mesh-closed", choices=["on", "off"], default="off")
    r.add_argument("--check-mesh-manifold", choices=["on", "off"], default="off")
    r.add_argument("--check-mesh-orientation", choices=["on", "off"], default="off")
    r.add_argument("--check-mesh-debug", choices=["on", "off"], default="off")
    r.add_argument("-q", "--quiet", action="store_true")
    r.add_argument("-v", action="count", default=0)
    r.add_argument("--device", type=int, default=None)                               # CUDA device of this process (default: LOCAL_RANK or 0)
    r.add_argument("--partition", choices=["on", "off"], default="off")              # under a multi-process launcher: ONE frame over all GPUs (slab partition)
    # anisotropic kernels (Yu & Turk 2013), an extension of this package: DESIGN.md "Anisotropic kernels"
    r.add_argument("--anisotropic", choices=["on", "off"], default="off")
    r.add_argument("--anisotropy-max-ratio", type=float, default=4.0)
    r.add_argument("--anisotropy-min-neighbors", type=int, default=10)
    r.add_argument("--anisotropy-smoothing", type=float, default=0.9)
    r.add_argument("--shard", default=None, metavar="I/N")                           # this process takes frames I, I + N, ... (default: RANK / WORLD_SIZE)
    # `splashsurf convert` (splashsurf/src/convert.rs:13-56)
    cv = sub.add_parser("convert")
    cv.add_argument("--particles", dest="input_particles", default=None)
    cv.add_argument("--mesh", dest="input_mesh", default=None)
    cv.add_argument("-o", dest="output_file", required=True)
    cv.add_argument("--overwrite", action="store_true")
    cv.add_argument("--domain-min", type=float, nargs=3, default=None, metavar=("X_MIN", "Y_MIN", "Z_MIN"))
    cv.add_argument("--domain-max", type=float, nargs=3, default=None, metavar=("X_MAX", "Y_MAX", "Z_MAX"))
    a = ap.parse_args(argv)
    if a.cmd == "convert":
        return convert(a)
    return reconstruct(a)


def collect_paths(a):
    """`ReconstructionRunnerPathCollection` (reconstruct.rs:700-963): the (input, output) pairs of one command line.  A "{}" in the
    input file name makes it a sequence: every file of that directory whose name matches prefix + digits + suffix and whose index lies in
    [--start-index, --end-index], in natural order; the output name needs a "{}" too (default "<stem with {} -> surface_{}>.vtk").  A
    single file defaults to "<stem>_surface.vtk".  --output-dir is prepended and created when missing."""
    import os
    import re
    inp = a.input
    name = os.path.basename(inp)
    if not name:
        raise ValueError(f'The input file path "{inp}" does not end with a filename')
    parent = os.path.dirname(inp)
    if parent and not os.path.isdir(parent):
        raise ValueError(f'The parent directory "{parent}" of the input file path "{inp}" does not exist')
    seq = "{}" in name
    stem = os.path.splitext(name)[0]
    if seq:
        if a.output_file is not None:
            if "{}" not in a.output_file:
                raise ValueError(f'The output filename "{a.output_file}" does not contain a place holder "{{}}"')
            out = a.output_file
        else:
            out = stem.replace("{}", "surface_{}") + ".vtk"
    else:
        if not os.path.isfile(inp):
            raise ValueError(f'Input file does not exist: "{inp}"')
        out = a.output_file if a.output_file is not None else f"{stem}_surface.vtk"
    if a.start_index is not None and a.end_index is not None and a.start_index > a.end_index:
        raise ValueError(f'Invalid input sequence range: "{a.start_index} to {a.end_index}"')
    if a.output_dir is not None:
        out = os.path.join(a.output_dir, out)
        d = os.path.dirname(out)
        if d and not os.path.exists(d):
            os.makedirs(d, exist_ok=True)
    if not seq:
        return [(inp, out)]
    prefix, suffix = name.split("{}", 1)
    rx = re.compile(re.escape(prefix) + r"(\d+)" + re.escape(suffix))          # unanchored, like Regex::is_match
    out_dir, out_pat = os.path.dirname(out), os.path.basename(out)

    def natural(n):
        return [(0, int(t)) if t.isdigit() else (1, t.lower()) for t in re.split(r"(\d+)", n) if t]
    paths = []
    for entry in sorted(os.listdir(parent or "."), key=natural):
        m = rx.search(entry)
        if m is None or not os.path.isfile(os.path.join(parent or ".", entry)):
            continue
        idx = int(m.group(1))
        if (a.start_index is not None and idx < a.start_index) or (a.end_index is not None and idx > a.end_index):
            continue
        paths.append((os.path.join(parent, entry), os.path.join(out_dir, out_pat.replace("{}", m.group(1)))))
    return paths


def _aabb(lo, hi, what):
    if (lo is None) != (hi is None):
        raise ValueError(f"the {what} needs both its min and its max corner")
    if lo is None:
        return None, None
    if any(h < l for l, h in zip(lo, hi)):
        raise ValueError(f"The user specified {what} min/max values are inconsistent! min: {list(lo)} max: {list(hi)}")
    if any(h == l for l, h in zip(lo, hi)):
        raise ValueError(f"The user specified {what} is degenerate! min: {list(lo)} max: {list(hi)}")
    return list(lo), list(hi)


def reconstruct_partitioned(a, paths) -> int:
    """--partition=on under torchrun: every frame is reconstructed by ALL processes together (slab partition of the subdomain grid, one
    halo exchange, mesh assembled on rank 0: splashsurf_b200.distributed) -- for clouds that are too large or too slow for one GPU.  Every
    rank reads its contiguous share of the particles; rank 0 writes the mesh.  The mesh post-processing steps are single-GPU steps and are
    refused here, except SPH normals (--normals=on --sph-normals=on), which travel with the assembled mesh."""
    import os
    import torch.distributed as dist
    from . import io
    from .distributed import DistributedReconstructor
    on = lambda v: str(v).lower() == "on"         # noqa: E731
    sph = on(a.normals) and on(a.sph_normals)
    refused = [k for k, v in (("-a", bool(a.interpolate_attributes)), ("--normals without --sph-normals", on(a.normals) and not sph),
                              ("--mesh-cleanup", on(a.mesh_cleanup or "off")), ("--decimate-barnacles", on(a.decimate_barnacles)),
                              ("--mesh-smoothing-iters", a.mesh_smoothing_iters is not None), ("--generate-quads", on(a.generate_quads)),
                              ("--mesh-aabb-min", a.mesh_aabb_min is not None), ("--normals-smoothing-iters", a.normals_smoothing_iters is not None)) if v]
    if refused:
        raise ValueError("--partition=on reconstructs without mesh post-processing; not available: " + ", ".join(refused))
    if not dist.is_initialized():
        dist.init_process_group(os.environ.get("SS_DIST_BACKEND", "nccl"))
    rank, world = dist.get_rank(), dist.get_world_size()
    pmin, pmax = _aabb(a.particle_aabb_min, a.particle_aabb_max, "particle AABB")
    rec = DistributedReconstructor(sph_normals=sph, device=os.environ.get("SS_RUNNER_DEVICE") or None, particle_radius=a.particle_radius,
                                   rest_density=a.rest_density, smoothing_length=a.smoothing_length, cube_size=a.cube_size,
                                   iso_surface_threshold=a.surface_threshold, simd=on(a.simd), subdomain_grid=on(a.subdomain_grid),
                                   subdomain_grid_auto_disable=not on(a.subdomain_grid_auto_disable), subdomain_num_cubes_per_dim=a.subdomain_cubes,
                                   aabb_min=pmin, aabb_max=pmax)
    try:
        for k, (src, dst) in enumerate(paths):
            p = io.read_particles(src)
            n = len(p)
            t = time.perf_counter()
            out = rec(p[(n * rank) // world:(n * (rank + 1)) // world])
            dt = time.perf_counter() - t
            if rank == 0:
                if not a.quiet:
                    print(f"[{k + 1}/{len(paths)}] {src}: {n} particles on {world} GPUs -> {out.nvertices} vertices, {out.ncells} triangles in {dt:.3f} s",
                          file=sys.stderr)
                if dst.endswith(".npz"):
                    np.savez(dst, vertices=out.mesh.vertices, triangles=out.mesh.triangles, **out.point_attributes)
                else:
                    io.write_mesh(dst, out)
    finally:
        rec.close()
    return 0


def reconstruct(a) -> int:
    """`reconstruct_subcommand` (reconstruct.rs:380-440, :1590-1680): one reconstruction (+ post-processing) per input file, the frames of
    a sequence one after the other on one context (its device buffers are reused from frame to frame).  Under a multi-process launcher
    (RANK / WORLD_SIZE / LOCAL_RANK in the environment, or --shard i/n) every process takes every n-th frame on its own GPU -- the device
    version of the reference's --mt-files; no collective is involved."""
    import os
    from . import Context, MeshWithData, io, reconstruct_surface, reconstruction_pipeline
    on = lambda v: str(v).lower() == "on"         # noqa: E731
    if on(a.double_precision):
        raise ValueError("--double-precision=on: the device path reconstructs float32 particles only (SURVEY.md 8b)")
    if on(a.partition) and on(a.anisotropic):
        raise ValueError("--partition=on does not support --anisotropic=on: the halo exchange does not carry the kernel centres")
    paths = collect_paths(a)
    if on(a.partition) and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        return reconstruct_partitioned(a, paths)
    rank, world = 0, 1
    if a.shard:
        rank, world = (int(t) for t in a.shard.split("/"))
    elif "WORLD_SIZE" in os.environ and int(os.environ["WORLD_SIZE"]) > 1:
        rank, world = int(os.environ.get("RANK", "0")), int(os.environ["WORLD_SIZE"])
    if not (0 <= rank < world):
        raise ValueError(f"invalid shard {rank}/{world}")
    paths = paths[rank::world]
    device = a.device if a.device is not None else int(os.environ.get("LOCAL_RANK", "0"))
    pmin, pmax = _aabb(a.particle_aabb_min, a.particle_aabb_max, "particle AABB")
    mmin, mmax = _aabb(a.mesh_aabb_min, a.mesh_aabb_max, "mesh AABB")
    # auto_disable is inverted in the reference CLI (reconstruct.rs:635; SURVEY.md 8b): with the defaults the subdomain grid is always used
    base = dict(particle_radius=a.particle_radius, rest_density=a.rest_density, smoothing_length=a.smoothing_length, cube_size=a.cube_size,
                iso_surface_threshold=a.surface_threshold, simd=on(a.simd), subdomain_grid=on(a.subdomain_grid),
                subdomain_grid_auto_disable=not on(a.subdomain_grid_auto_disable), subdomain_num_cubes_per_dim=a.subdomain_cubes,
                aabb_min=pmin, aabb_max=pmax, multi_threading=on(a.mt_particles), anisotropic=on(a.anisotropic),
                anisotropy_max_ratio=a.anisotropy_max_ratio, anisotropy_min_neighbors=a.anisotropy_min_neighbors,
                anisotropy_smoothing=a.anisotropy_smoothing)
    if a.mesh_cleanup is None:
        a.mesh_cleanup = "on" if a.mesh_smoothing_iters not in (None, 0) else "off"
    chk = on(a.check_mesh)
    closed, manifold, orient = chk or on(a.check_mesh_closed), chk or on(a.check_mesh_manifold), chk or on(a.check_mesh_orientation)
    post = any([bool(a.interpolate_attributes), on(a.normals), on(a.mesh_cleanup), on(a.decimate_barnacles), a.mesh_smoothing_iters is not None,
                on(a.generate_quads), mmin is not None, closed, manifold, orient])
    ctx = Context(device) if paths else None
    try:
        for k, (src, dst) in enumerate(paths):
            p = io.read_particles(src)
            attrs = io.read_particle_attributes(src, a.interpolate_attributes)
            for name, arr in attrs.items():
                if arr.dtype.kind != "f":              # BGEO Int attributes load as u64; the reference cannot interpolate them either (reconstruct.rs:1387)
                    raise ValueError(f'Interpolation of this attribute type not implemented (attribute "{name}")')
            t = time.perf_counter()
            if post:
                # --sph-normals only selects how --normals are computed (reconstruct.rs:1094-1149)
                out, rec = reconstruction_pipeline(
                    p, attributes_to_interpolate=attrs, compute_normals=on(a.normals), sph_normals=on(a.sph_normals),
                    normals_smoothing_iters=a.normals_smoothing_iters, mesh_smoothing_iters=a.mesh_smoothing_iters,
                    mesh_smoothing_weights=on(a.mesh_smoothing_weights), mesh_smoothing_weights_normalization=a.mesh_smoothing_weights_normalization,
                    output_mesh_smoothing_weights=on(a.output_smoothing_weights), output_raw_normals=on(a.output_raw_normals),
                    mesh_cleanup=on(a.mesh_cleanup), mesh_cleanup_snap_dist=a.mesh_cleanup_snap_dist, decimate_barnacles=on(a.decimate_barnacles),
                    keep_vertices=on(a.keep_verts), generate_quads=on(a.generate_quads), quad_max_edge_diag_ratio=a.quad_max_edge_diag_ratio,
                    quad_max_normal_angle=a.quad_max_normal_angle, quad_max_interior_angle=a.quad_max_interior_angle, mesh_aabb_min=mmin,
                    mesh_aabb_max=mmax, mesh_aabb_clamp_vertices=on(a.mesh_aabb_clamp_verts), check_mesh_closed=closed, check_mesh_manifold=manifold,
                    check_mesh_orientation=orient, check_mesh_debug=on(a.check_mesh_debug), context=ctx, **base)
                raw = rec.mesh
            else:
                raw = reconstruct_surface(p, context=ctx, **base).mesh
                out = MeshWithData(raw, {}, {})
            dt = time.perf_counter() - t
            quads = out.mesh.get_quads() if on(a.generate_quads) else None
            tris = out.mesh.get_triangles() if on(a.generate_quads) else out.mesh.triangles
            if not a.quiet:
                print(f"[{k + 1}/{len(paths)}] {src}: {len(p)} particles -> {out.nvertices} vertices, {len(tris)} triangles"
                      + (f", {len(quads)} quads" if quads is not None else "") + f" in {dt:.3f} s", file=sys.stderr)
            t = time.perf_counter()
            if on(a.output_raw_mesh):                  # "raw_" + file name beside the output file (reconstruct.rs:1618-1650)
                io.write_mesh(os.path.join(os.path.dirname(dst), "raw_" + os.path.basename(dst)), MeshWithData(raw, {}, {}))
            if dst.endswith(".npz"):
                np.savez(dst, vertices=out.mesh.vertices, triangles=tris, **({"quads": quads} if quads is not None else {}), **out.point_attributes)
            else:
                io.write_mesh(dst, out)                # .vtk / .ply / .obj as the reference CLI writes them (io.rs:276-316)
            if not a.quiet:
                print(f"wrote {dst} in {time.perf_counter() - t:.3f} s", file=sys.stderr)
    finally:
        if ctx is not None:
            ctx.close()
    return 0


def _entry() -> int:
    """Process entry point: errors become one line on stderr and exit code 1 (the reference binary logs `Error occurred: ...`)."""
    from . import SplashsurfError
    try:
        return main()
    except (ValueError, OSError, SplashsurfError, NotImplementedError) as e:
        print(f"Error occurred: {e}", file=sys.stderr)
        return 1


if __name__ == "__main__":
    sys.exit(_entry())
