"""Isotropic vs anisotropic reconstruction on bench.py's flagship cloud (synthetic 50 M-particle dam break, r = 0.01, l = 2, c = 0.5,
threshold 0.6), alternating the two in one process on one context, timed with device events around whole calls (particles
already on the device), plus the stage times the library reports.  Writes one JSON file (default
profiles/r3_bench_anisotropic.json) with the card's name and power limit read in the same run.

    python tools/bench_anisotropic.py [--particles N] [--steps K] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import splashsurf_b200 as ss  # noqa: E402
from splashsurf_b200 import synthetic as syn  # noqa: E402

KW = dict(particle_radius=0.01, smoothing_length=2.0, cube_size=0.5, iso_surface_threshold=0.6)
STAGES = ("decomposition", "density", "binning", "tile_setup", "levelset", "marching_cubes", "stitching", "total_device")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi unavailable)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=0, help="0: the 50 M flagship cloud; else a dam break scaled to about N")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_anisotropic.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    p = syn.dam_break_50m() if a.particles == 0 else syn.dam_break_scaled(a.particles, 0.01, 3)
    dev = torch.from_numpy(p).cuda()
    ctx = ss.Context(0)
    L = ctx._L
    prm = ss.make_params(**KW)
    runs = {"isotropic": [], "anisotropic": []}

    def one(aniso):
        ss._set_anisotropy(ctx, aniso, 4.0, 10, 0.9)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        s = ctx.reconstruct_raw(dev.data_ptr(), len(p), prm)
        e1.record()
        torch.cuda.synchronize()
        try:
            tm = ctx.timings(s)
            rec = {"call_ms": e0.elapsed_time(e1), "vertices": L.ss_surface_num_vertices(s), "triangles": L.ss_surface_num_triangles(s)}
            rec.update({k: tm[k] for k in STAGES})
            if aniso:
                ms, sw = (ss.C.c_float * 2)(), ss.C.c_uint32()
                ss._check(L, L.ss_surface_anisotropy_stats(s, ms, ss.C.byref(sw)))
                rec.update(anisotropy_moments=ms[0], anisotropy_decomposition=ms[1], anisotropy_max_jacobi_sweeps=sw.value)
            return rec
        finally:
            ctx.free_surface(s)
            ss._set_anisotropy(ctx, False, 4.0, 10, 0.9)

    one(False)
    one(True)                       # warm-up of both shapes
    for _ in range(a.steps):
        for mode in (False, True):
            runs["anisotropic" if mode else "isotropic"].append(one(mode))
    med = {k: {f: float(np.median([r[f] for r in v])) for f in v[0]} for k, v in runs.items()}
    out = {"card": card(), "particles": int(len(p)), "params": KW, "anisotropy": {"max_ratio": 4.0, "min_neighbors": 10, "smoothing": 0.9},
           "steps": a.steps, "median": med, "runs": runs, "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"card": out["card"], "particles": out["particles"], "median": med}))
    ctx.close()


if __name__ == "__main__":
    main()
