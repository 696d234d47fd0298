#!/usr/bin/env python3
"""bench.py -- Mparticles/s of the reconstruct hot path (BASELINE.json metric) on N B200s of one node.

A step = one full `reconstruct_surface` pass (decomposition -> densities -> level-set splat -> marching cubes ->
stitching) over one synthetic particle cloud.  Workload at N=1: BASELINE configs[3], the 50 M-particle dam break the
metric is quoted on (it fits one B200).  `value` is timed with the particles already resident in HBM (CUDA events on
the library's stream around every step); `e2e` runs the same call through the C ABI with HOST buffers -- pinned input
copied host->device and the mesh copied device->host inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--particles M] [--impl reference]
                  [--workload cfg2|cfg3|cfg4|cfg5|cfg5_overlap] [--levelset-variant 0|1|2] [--density-variant 0|1|2] [--mc-variant 0|1]
                  [--runner-protocol stats|two_call|callback] [--sph-normals] [--no-cpu-baseline] [--no-extra-e2e]
                  [--dump-outputs DIR]

(The defaults are the measured configuration: level-set variant 2, density variant 0, marching-cubes variant 1, "stats" runner
protocol.  tests/test_bench_dry_run.py runs this file's main() on the CPU executor of the CUDA sources to check its control flow
and the JSON contract.)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mparticles/s end-to-end reconstruct (50M pts, cell=0.5r) at 1/2/4/8 GPU vs CPU ref"     # BASELINE.json
RECON_KW = dict(particle_radius=0.01, smoothing_length=2.0, cube_size=0.5, iso_surface_threshold=0.6)
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 flop x max SM clock (nominal)


def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index="0"):
        self.rows, self.proc, self.gpu, self.first = [], None, gpu_index, 0

    def mark(self):
        """Start of the timed region: only samples taken from here on are reported (the process itself is started before the
        warm-up, so that NVML's start-up on a multi-GPU box does not fall into the timed steps)."""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows[self.first:]:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


WORKLOADS = {
    "cfg4": None,    # default: dam break (50 M, or scaled with --particles)
    "cfg2": ("synthetic jittered cube 100^3 = 1 M particles (r=0.025, seed 1234)", dict(particle_radius=0.025)),
    "cfg3": ("synthetic dam-break 10 M (column 200x230x200 + sheet 400x10x200, r=0.01, seed 2)", dict()),
    "cfg5": ("synthetic splash 200 M (body 540x583x540 + ~340 disjoint droplets of radius 10..40 d above it, r=0.005, seed 4), cube 0.45 r",
             dict(particle_radius=0.005, cube_size=0.45)),
    # the round-2 first-run cloud: droplet lattices superimposed at 2-3x rest density (stress case for the dense-cluster routes)
    "cfg5_overlap": ("synthetic splash 200 M with superimposed droplets (body 540x583x540, r=0.005, seed 4), cube 0.45 r",
                     dict(particle_radius=0.005, cube_size=0.45)),
}


def make_cloud(n_target, workload="cfg4"):
    from splashsurf_b200 import synthetic as syn
    if workload == "cfg2":
        return syn.jittered_cube(100, 0.025, 1234), WORKLOADS["cfg2"][0]
    if workload == "cfg3":
        return syn.dam_break_10m(), WORKLOADS["cfg3"][0]
    if workload in ("cfg5", "cfg5_overlap"):
        return syn.splash_200m(overlap=workload == "cfg5_overlap"), WORKLOADS[workload][0]
    if n_target >= 50_000_000:
        return syn.dam_break_50m(), "synthetic dam-break 50 M (column 340x370x340 + sheet 1063x20x340, r=0.01, seed 3)"
    return syn.dam_break_scaled(n_target, 0.01, 3), f"synthetic dam-break scaled to ~{n_target} particles (cfg-4 proportions, r=0.01, seed 3)"


def time_reference(p, repeats, kw=None):
    """The reference's own CPU implementation (pysplashsurf 0.14.0 wheel, rayon + AVX2) on all host cores."""
    import oracle
    ps = oracle.reference()
    kw = kw or RECON_KW
    best = None
    for _ in range(repeats):
        t = time.perf_counter()
        r = ps.reconstruct_surface(p, particle_radius=kw["particle_radius"], smoothing_length=kw["smoothing_length"],
                                   cube_size=kw["cube_size"], iso_surface_threshold=kw["iso_surface_threshold"],
                                   multi_threading=True, simd=True, subdomain_grid=True, subdomain_num_cubes_per_dim=64)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
        nv, nt = len(r.mesh.vertices), len(r.mesh.triangles)
        del r
    return best, nv, nt


def cpu_stage_tree(p, kw):
    """Per-stage wall times of the reference CLI pipeline (`splashsurf reconstruct -v`, cli.rs:124-130, README.md:198-231) on
    the particle set `p`, parsed from the profile tree it logs.  Runs in a child process (the tree goes to the child's stderr).
    Returns {} when anything goes wrong -- it is a side-by-side diagnostic, never part of a timed region."""
    import re, tempfile
    try:
        d = tempfile.mkdtemp(prefix="ss_stage_")
        xyz = os.path.join(d, "cloud.xyz")
        np.ascontiguousarray(p, dtype="<f4").tofile(xyz)
        code = ("import sys; sys.path.insert(0, %r); import oracle; ps = oracle.reference(); "
                "ps.run_splashsurf(['splashsurf', 'reconstruct', %r, '-r=%r', '-l=%r', '-c=%r', '-t=%r', '-o', %r, '-v'])"
                % (ROOT, xyz, kw["particle_radius"], kw["smoothing_length"], kw["cube_size"], kw["iso_surface_threshold"], os.path.join(d, "out.vtk")))
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
        out = {}
        want = {"surface reconstruction subdomain-grid": "total", "decomposition": "decomposition", "compute_global_density_vector": "density",
                "reconstruction": "levelset_plus_marching_cubes", "stitching": "stitching",
                "density grid loop (avx)": "levelset_dense_cpu_seconds_summed", "density grid loop (sparse)": "levelset_sparse_cpu_seconds_summed",
                "mc triangulation loop": "marching_cubes_cpu_seconds_summed"}
        for line in (res.stdout + "\n" + res.stderr).splitlines():
            m = re.search(r"\]\s+([^:\]]+?): [^,]*, ([0-9.]+)ms avg, (\d+) calls? \(total: ([0-9.]+)s\)", line)
            if not m:
                continue
            name, avg_ms, calls, total_s = m.group(1).strip(), float(m.group(2)), int(m.group(3)), float(m.group(4))
            key = want.get(name)
            if key is None:
                continue
            if key.endswith("_summed"):
                out[key] = out.get(key, 0.0) + total_s
            elif key not in out:
                out[key] = avg_ms if calls == 1 else total_s * 1e3
        for f in os.listdir(d):
            os.remove(os.path.join(d, f))
        os.rmdir(d)
        return out
    except Exception as e:      # noqa: BLE001
        return {"error": str(e)[:200]}


DUMP_MAX_ROWS = 1 << 20      # per array: vertices 12 MB (f32), triangles 24 MB (f64), normals 12 MB -> under 64 MB in all


def canonical_mesh(vertices, triangles, normals=None):
    """The mesh in an order that does not depend on the order the library emits it in: vertices sorted by position (then normal),
    triangles renumbered (coincident vertices take the number of the first of them), rotated to their lexicographically smallest
    rotation and sorted.  Two builds that compute the same mesh write the same arrays, and sampled rows of them are the same rows."""
    v = np.asarray(vertices, np.float32).reshape(-1, 3)
    keys = [v[:, 2], v[:, 1], v[:, 0]]
    if normals is not None:
        keys = [normals[:, 2], normals[:, 1], normals[:, 0]] + keys
    order = np.lexsort(keys)
    vs = v[order]
    first = np.r_[True, (vs[1:] != vs[:-1]).any(axis=1)] if len(vs) else np.zeros(0, bool)
    start = np.maximum.accumulate(np.where(first, np.arange(len(vs)), 0))        # sorted index of the first coincident vertex
    number = np.empty(len(v), np.int64)
    number[order] = start
    t = number[np.asarray(triangles).astype(np.int64).reshape(-1, 3)]
    if len(t):
        best = t.copy()
        for r in (t[:, [1, 2, 0]], t[:, [2, 0, 1]]):
            less = (r[:, 0] < best[:, 0]) | ((r[:, 0] == best[:, 0]) & ((r[:, 1] < best[:, 1]) | ((r[:, 1] == best[:, 1]) & (r[:, 2] < best[:, 2]))))
            best[less] = r[less]
        t = best[np.lexsort((best[:, 2], best[:, 1], best[:, 0]))]
    return vs, t, (None if normals is None else np.asarray(normals)[order])


def dump_outputs(out_dir, arrays):
    """Writes arrays as <out_dir>/<name>.npy (float32 or float64).  An array of more than DUMP_MAX_ROWS rows is reduced to a
    fixed sample of rows (seed 0, ascending row order): with arrays in canonical order (canonical_mesh), two builds given the
    same arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if len(a) > DUMP_MAX_ROWS:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), DUMP_MAX_ROWS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(args, desc, n_total, kw, parallelism):
    wl = args.workload
    return {"workload": (wl + ": " if wl != "cfg4" else ("cfg-4: " if n_total >= 50_000_000 else "cfg-4 (scaled): ")) + desc,
            "particles": int(n_total), "r": kw["particle_radius"], "cube_size": f"{kw['cube_size']}r", "smoothing_length": "2.0r", "iso": 0.6,
            "subdomain_cubes": 64, "parallelism": parallelism}


def run_reference(args):
    """The reference's own CPU implementation on the SAME cloud as the b200 arm (every step = one full reconstruct_surface of
    the whole workload, all host threads).  `--ref-particles N` is an explicit opt-out (bounded sample, flagged in config)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle
    kw = dict(RECON_KW)
    if WORKLOADS.get(args.workload):
        kw.update(WORKLOADS[args.workload][1])
    bounded = args.ref_particles is not None
    p, desc = make_cloud(args.ref_particles if bounded else args.particles, args.workload)
    if not oracle.reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref (reference wheel) not present on this box"}))
        return 0
    budget_s = float(os.environ.get("SS_REF_BUDGET_S", "700"))   # SCALE_r01 ran every N under an 870 s limit
    t_start = time.perf_counter()
    times, warm_done, nv, nt = [], 0, 0, 0
    steps, warmup = args.steps, args.warmup
    for i in range(args.warmup + args.steps):
        dt, nv, nt = time_reference(p, 1, kw)
        if i < warmup:
            warm_done += 1
        else:
            times.append(dt)
        # budget guard: the whole arm has to end within the driver's limit even on a slow host; drop warm-ups first, then steps
        left = budget_s - (time.perf_counter() - t_start)
        if i + 1 < warmup and (warmup - i - 1 + steps) * dt > left:
            warmup = i + 1
        if len(times) >= 1 and (steps - len(times)) * dt > left:
            break
    ms = 1e3 * float(np.mean(times))
    val = len(p) / (ms * 1e-3) / 1e6
    cfg = workload_config(args, desc, len(p), kw, f"rayon, {os.cpu_count()} host threads")
    cfg["bounded_sample"] = bool(bounded)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mparticles/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": warm_done, "steps_requested": args.steps, "warmup_requested": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": val, "unit": "Mparticles/s", "cores": os.cpu_count(), "kind": "reference",
                             "sample": f"all {len(p)} particles of the workload per step, pysplashsurf 0.14.0 wheel (portable manylinux build, runtime AVX2), all host threads"},
            "e2e": {"value": val, "unit": "Mparticles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "mesh": {"vertices": nv, "triangles": nt}}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--particles", type=int, default=50_000_400, help="target particle count of the dam break (default: cfg-4)")
    ap.add_argument("--ref-particles", type=int, default=None,
                    help="--impl reference only: time a bounded sample of this many particles instead of the whole workload (opt-out, flagged)")
    ap.add_argument("--cpu-sample-particles", type=int, default=2_000_000, help="size of the bounded sample of the cpu_baseline leg")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS), help="BASELINE config (default cfg4 = the metric's 50 M dam break)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sph-normals", action="store_true", help="also compute SPH normals at the mesh vertices (cfg-5; sph_interpolation.rs:82-133)")
    ap.add_argument("--runner-protocol", default="stats", choices=["stats", "two_call", "callback"],
                    help="multi-GPU only: how the global subdomain maximum reaches the library (see distributed.Runner)")
    ap.add_argument("--levelset-variant", type=int, default=2, choices=[0, 1, 2],
                    help="2 (default): warp-per-brick certification + exact kernels (TMA staging, packed FP32); 1: CTA-per-brick certification kernel; 0: fused k_levelset")
    ap.add_argument("--no-extra-e2e", action="store_true", help="skip the e2e_frontend reading (one GPU only)")
    ap.add_argument("--density-variant", type=int, default=0, choices=[0, 1, 2], help="0 (default): thread per particle; 1 / 2: cell-cooperative density kernel (staging by bulk copies / loads; slower)")
    ap.add_argument("--mc-variant", type=int, default=1, choices=[0, 1], help="1 (default): warp-per-brick marching cubes / fix-up sweep; 0: CTA per brick")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the mesh of the last timed step to DIR/*.npy in canonical order (vertices sorted by position, triangles "
                         "renumbered and sorted; mesh_counts; normals with --sph-normals on several GPUs); arrays above %d rows are a "
                         "fixed sample of rows" % DUMP_MAX_ROWS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.impl == "reference":
        return run_reference(args)
    # stdout hygiene: NCCL / library chatter must not precede the JSON line -> fd 1 points at stderr until the end
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the reconstruct path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        # a mismatched collective must fail fast instead of burning the default 10-minute NCCL timeout
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=240))

    import splashsurf_b200 as ss
    from splashsurf_b200 import distributed as ssd
    ctx = ss.Context(local_rank)
    ctx.set_levelset_variant(args.levelset_variant)
    ctx.set_density_variant(args.density_variant)
    ctx.set_mc_variant(args.mc_variant)
    if args.sph_normals:
        ss._check(ctx._L, ctx._L.ss_context_set_compute_sph_normals(ctx._h, 1))
    kw = dict(RECON_KW)
    if WORKLOADS.get(args.workload):
        kw.update(WORKLOADS[args.workload][1])
    params = ss.make_params(**kw)

    # ---- workload (identical on every rank; each rank keeps its slab when world > 1)
    p_all, desc = make_cloud(args.particles, args.workload)
    n_total = len(p_all)
    runner = ssd.Runner(ctx, params, world, rank, local_rank, protocol=args.runner_protocol)
    runner.ctx_normals = bool(args.sph_normals)
    p_local = runner.take_local(p_all)
    del p_all
    host_in = torch.from_numpy(p_local).pin_memory()
    dev_in = host_in.cuda(non_blocking=False)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident steps
    # one nvidia-smi process (rank 0) watches every GPU of the job; started before the warm-up, read from the timed region on
    sampler = ClockSampler(",".join(str(g) for g in range(world)) if world > 1 else str(local_rank))
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        res = runner.step(dev_in, copy_out=False)
    # The multi-GPU runner tunes its slab cuts from the measured per-rank times of the first frames and then keeps the best plan
    # (a simulation feeds it thousands of frames).  A short warm-up can end before that: run untimed settling steps until the plan
    # stands still, plus one for the buffers of the final cuts -- the timed region then measures the steady state.  Counted and
    # reported (`config.plan_settling_steps`); the same number on every rank, the decision comes from all-reduced times.
    settling = 0
    while world > 1 and not runner.plan_settled and settling < 8:
        res = runner.step(dev_in, copy_out=False)
        settling += 1
    if settling:
        res = runner.step(dev_in, copy_out=False)
        settling += 1
    barrier()
    sampler.mark()
    dev_ms, ls_ms, launches, pairs, ls_launches = 0.0, 0.0, 0, 0.0, 0
    step_ms = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        # --dump-outputs: the last timed step also copies its mesh to the host (after the step's device timing has been taken)
        res = runner.step(dev_in, copy_out=bool(args.dump_outputs) and i == args.steps - 1)
        dev_ms += res["device_ms"]; ls_ms += res["timings"]["levelset"]; launches += res["launches"]; step_ms.append(round(res["device_ms"], 2))
        pairs += res["timings"]["levelset_pairs"]; ls_launches += res["timings"]["levelset_launches"]
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        nv_d, nt_d = (res["nv"], res["nt"]) if world == 1 else (res["nv_global"], res["nt_global"])
        v_d, t_d, n_d = canonical_mesh(*runner.gathered_mesh(nv_d, nt_d), runner.gathered_normals())
        dumped = {"vertices": v_d, "triangles": t_d, "mesh_counts": np.array([nv_d, nt_d], np.float64)}
        if n_d is not None:
            dumped["normals"] = n_d
        dump_outputs(args.dump_outputs, dumped)
    sys.stderr.write(f"[rank {rank}] device ms/step {dev_ms / args.steps:.2f}, level-set {ls_ms / args.steps:.2f}, particles processed {res.get('recv_particles', len(p_local))}\n")
    stats = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    dev_ms_max, wall_ms_max = stats.tolist()
    ms_per_step = dev_ms_max / args.steps
    value = n_total / (ms_per_step * 1e-3) / 1e6
    agg = torch.tensor([res["nv"], res["nt"], res["nsub_owned"], res["memberships"], ls_ms, pairs, float(launches)], dtype=torch.float64, device="cuda")
    if world > 1:
        agg_max = agg.clone()
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
        dist.all_reduce(agg_max, op=dist.ReduceOp.MAX)
        ls_ms = float(agg_max[4])            # slowest rank's level-set time
    nv, nt, nsub_total, memberships_total = int(agg[0]), int(agg[1]), int(agg[2]), float(agg[3])
    launches = int(agg[6])
    # one instrumented step (outside the timed region) for the work model of the level-set kernel
    ctx.set_count_pairs(True)
    tm_c = runner.step(dev_in, copy_out=False)["timings"]
    pairs_t = torch.tensor([tm_c["levelset_pairs"] * args.steps, tm_c.get("levelset_cert_evals", 0.0) * args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(pairs_t, op=dist.ReduceOp.SUM)
    pairs, cert_evals = float(pairs_t[0].item()), float(pairs_t[1].item())
    ctx.set_count_pairs(False)
    fixups = res["timings"].get("levelset_fixup_points", 0)
    stage = {k: round(v, 3) for k, v in res["timings"].items() if isinstance(v, float)}
    bricks = {k: int(v) for k, v in res["timings"].items() if k.startswith("bricks_")}
    if res.get("phase_ms"):
        sys.stderr.write(f"[rank {rank}] runner phases of the last step (host ms): {res['phase_ms']}\n")

    # ---- end to end through the C ABI with host buffers (pinned input, mesh copied back)
    for _ in range(min(args.warmup, 2)):
        runner.step(host_in, copy_out=True)
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    nv_g = nt_g = None
    for _ in range(args.steps):
        r2 = runner.step(host_in, copy_out=True)
        d2h = r2["d2h_bytes"]
        if r2.get("nv_global") is not None:
            nv_g, nt_g = r2["nv_global"], r2["nt_global"]
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
    tb = torch.tensor([float(d2h)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tb, op=dist.ReduceOp.SUM)            # every rank copies its own part of the mesh to the shared host segment
    e2e_ms = t.item() / args.steps
    d2h = int(tb.item())
    e2e_val = n_total / (e2e_ms * 1e-3) / 1e6

    # ---- one more end-to-end reading on one GPU (extra key; `e2e` above stays the pinned-buffer number through the runner):
    #   e2e_frontend -- the documented front-end call splashsurf_b200.reconstruct_surface(numpy array): pageable input, fresh numpy outputs
    # (A frame-sequence API with two frames in flight was measured in round 2 and removed again: the library's ~15 small read-backs
    #  per step queue behind the 1 GB mesh download on the copy engine, 225 ms per frame against 151 ms serial.)
    e2e_frontend = None
    if world == 1 and not args.no_extra_e2e:
        t_fe = []
        for _ in range(3):
            t0 = time.perf_counter()
            r_fe = ss.reconstruct_surface(p_local, context=ctx, **kw)
            t_fe.append(time.perf_counter() - t0)
        assert r_fe.mesh.nvertices == res["nv"]
        e2e_frontend = {"value": n_total / min(t_fe[1:]) / 1e6, "unit": "Mparticles/s", "ms_per_step": 1e3 * min(t_fe[1:]),
                        "note": "splashsurf_b200.reconstruct_surface(numpy): pageable host input, freshly allocated numpy outputs (vertices f32, triangles u64, densities), best of 2 after one warm call"}
        del r_fe
        # same call with the context's reusable page-locked result buffers (Context.reuse_host_buffers): no fresh pages, PCIe-speed copies
        ctx.reuse_host_buffers = True
        t_fe = []
        for _ in range(3):
            t0 = time.perf_counter()
            r_fe = ss.reconstruct_surface(p_local, context=ctx, **kw)
            t_fe.append(time.perf_counter() - t0)
        assert r_fe.mesh.nvertices == res["nv"]
        e2e_frontend["reuse_host_buffers"] = {"value": n_total / min(t_fe[1:]) / 1e6, "ms_per_step": 1e3 * min(t_fe[1:]),
                                              "note": "same call, result arrays are views of the context's page-locked buffers (overwritten by the next call)"}
        del r_fe
        ctx.reuse_host_buffers = False

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        n_sub = nsub_total
        np3 = 65 ** 3
        # algorithmic bytes of the level-set kernel per step: particle records (16 B pos+V, 4 B k_split, 4 B index) of every
        # membership once + one f32 tile write per subdomain (SURVEY.md 8d K3: 16 g N + 4 P N)
        ls_bytes = memberships_total * 24.0 + n_sub * np3 * 4.0
        ls_s = (ls_ms / args.steps) * 1e-3
        ach = ls_bytes / ls_s / 1e9 if ls_s > 0 else 0.0
        flops = (pairs / args.steps) * 30.0
        traffic, traffic_note = None, None
        from splashsurf_b200 import build as ssbuild
        src_sha, ls_sha = ssbuild.source_hash(), ssbuild.levelset_source_hash()
        try:
            # DRAM bytes of the level-set kernels of ONE step (certification + exact pass + fix-up pass) from an `ncu --set full`
            # capture of this very workload; only accepted when the level-set sources are the ones the capture was taken on
            tj = json.load(open(os.path.join(ROOT, "profiles", "levelset_traffic.json")))
            if tj.get("levelset_source_sha") != ls_sha:
                traffic_note = f"refused: profiles/levelset_traffic.json was captured on level-set sources {tj.get('levelset_source_sha')}, this build is {ls_sha}"
            elif tj.get("particles") != int(n_total) or tj.get("workload") != args.workload or world != 1:
                traffic_note = f"refused: capture was taken on {tj.get('workload')} / {tj.get('particles')} particles / 1 GPU, this run is {args.workload} / {n_total} / {world} GPU(s)"
            else:
                traffic = float(tj["dram_bytes_per_step"])
                traffic_note = tj.get("source", "")
        except Exception as e:      # noqa: BLE001
            traffic_note = f"no capture: {e}"
        ls_kernel = {2: "level-set stage: k_certify_warp + k_exact_warp", 1: "level-set stage: k_certify + k_levelset (fix mode)", 0: "k_levelset"}[int(args.levelset_variant)]
        roof = {"bound": "hbm", "kernel": ls_kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "traffic_note": traffic_note,
                "peak_source": peak_src, "launches_per_step": ls_launches / args.steps, "ms_per_step": ls_ms / args.steps,
                "algorithmic_bytes_per_step": ls_bytes,
                "note": "the ordered level-set gather is FP32-issue bound, not HBM bound (SURVEY.md 8d): see fp32",
                "fp32": {"achieved_tflops": flops / ls_s / 1e12 if ls_s > 0 else 0.0, "peak_tflops": FP32_PEAK_TFLOPS,
                         "frac": (flops / ls_s / 1e12) / FP32_PEAK_TFLOPS if ls_s > 0 else 0.0,
                         "model": "exactly evaluated in-support particle-gridpoint pairs x 30 flop", "pairs_per_step": pairs / args.steps,
                         "fixup_points_per_step": int(fixups),
                         # everything the level-set kernels evaluate: + the lower-bound evaluations of the certification pass
                         # (d^2 from the shared dx^2 + dy^2: 2 flop, cubic bound by Horner: 6, clamp: 1, volume-weighted sum: 2)
                         "cert_evals_per_step": cert_evals / args.steps,
                         "achieved_tflops_incl_certification": (flops + (cert_evals / args.steps) * 11.0) / ls_s / 1e12 if ls_s > 0 else 0.0,
                         "frac_incl_certification": ((flops + (cert_evals / args.steps) * 11.0) / ls_s / 1e12) / FP32_PEAK_TFLOPS if ls_s > 0 else 0.0}}
        line = {"metric": METRIC, "value": value, "unit": "Mparticles/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": dict(workload_config(args, desc, n_total, kw, f"subdomain slabs x{world}" if world > 1 else "single GPU"),
                               levelset_variant=int(args.levelset_variant), density_variant=int(args.density_variant), mc_variant=int(args.mc_variant),
                               sph_normals=bool(args.sph_normals), plan_settling_steps=int(settling),
                               l2="inputs (600 MB) and tiles (GBs) exceed the 126 MB L2; no flush needed"),
                "mesh": {"vertices": int(nv_g if nv_g is not None else nv), "triangles": int(nt_g if nt_g is not None else nt), "subdomains": int(n_sub)},
                "wall_ms_per_step": wall_ms_max / args.steps, "step_ms_rank0": step_ms, "stage_ms_last_step": stage, "bricks_last_step_rank0": bricks, "runner_phase_ms_last_step_rank0": res.get("phase_ms"),
                "e2e": {"value": e2e_val, "unit": "Mparticles/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(len(p_local) * 12 * world),
                        "d2h_bytes_per_step": int(d2h)},
                "e2e_frontend": e2e_frontend,
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "source_sha": src_sha, "levelset_source_sha": ls_sha}
        if not args.no_cpu_baseline and world == 1:
            try:
                import oracle
                if oracle.reference_available():
                    ps, _ = make_cloud(args.cpu_sample_particles, "cfg4")
                    dt, _, _ = time_reference(ps, 2, RECON_KW)
                    line["cpu_baseline"] = {"value": len(ps) / dt / 1e6, "unit": "Mparticles/s", "cores": os.cpu_count(), "kind": "reference",
                                            "sample": f"{len(ps)}-particle dam break (same generator), best of 2, pysplashsurf 0.14.0 wheel on all host threads"}
                    # stage by stage beside the GPU's stage_ms: the reference CLI's own profile tree on the same sample
                    line["cpu_stage_ms"] = dict(cpu_stage_tree(ps, RECON_KW), particles=int(len(ps)),
                                                note="wall ms of `splashsurf reconstruct -v` stages on the bounded sample; *_cpu_seconds_summed are summed over worker threads")
                    # the GPU on the very same sample, for a like-for-like stage comparison
                    rs = ss.reconstruct_surface(ps, context=ctx, **RECON_KW)
                    rs = ss.reconstruct_surface(ps, context=ctx, **RECON_KW)
                    line["gpu_stage_ms_same_sample"] = {k: round(float(v), 3) for k, v in rs.timings.items()
                                                        if k in ("decomposition", "density", "binning", "levelset", "marching_cubes", "stitching", "total_device", "upload")}
                else:
                    line["cpu_baseline"] = {"value": None, "unit": "Mparticles/s", "cores": os.cpu_count(), "kind": "reference", "sample": "oracle/_ref missing"}
            except Exception as e:   # the baseline must never take the bench line down
                line["cpu_baseline"] = {"value": None, "unit": "Mparticles/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e}"}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
