"""bench.py's b200 arm executed here, without a GPU: tests/emul/run_on_executor.py maps torch's CUDA entry points to host
equivalents and binds the library to the CPU executor of the CUDA sources, then calls bench.main() unchanged.  Checks the
control flow (single rank and two gloo ranks, every command-line switch) and the contract of the JSON line; the numbers are
meaningless and never recorded."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT, free_port

LAUNCHER = os.path.join(ROOT, "tests", "emul", "run_on_executor.py")
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "clocks", "e2e", "gpu_launches", "roofline"}


def _check_line(out: str, n_gpus: int, steps: int):
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out[-2000:]                     # exactly ONE line on stdout
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["metric"] == json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    assert d["n_gpus"] == n_gpus and d["steps"] == steps and d["higher_is_better"] is True and d["unit"] == "Mparticles/s"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert "workload" in d["config"] and "model" not in d["config"]
    return d


def _check_dump(dump_dir, d):
    """--dump-outputs: the mesh of the last timed step in canonical order, float32 / float64 arrays, counts equal to the JSON line's."""
    import numpy as np
    arrays = {f[:-4]: np.load(os.path.join(dump_dir, f)) for f in sorted(os.listdir(dump_dir))}
    assert set(arrays) == {"mesh_counts", "triangles", "vertices"}, set(arrays)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values()) and sum(a.nbytes for a in arrays.values()) <= 64 << 20
    nv, nt = d["mesh"]["vertices"], d["mesh"]["triangles"]
    assert arrays["mesh_counts"].tolist() == [nv, nt] and arrays["vertices"].shape == (nv, 3) and arrays["triangles"].shape == (nt, 3)
    assert arrays["triangles"].min() >= 0 and arrays["triangles"].max() < nv
    # canonical order: vertices sorted by position, triangles sorted
    v, t = arrays["vertices"], arrays["triangles"]
    assert np.array_equal(np.lexsort(v.T[::-1]), np.arange(len(v))) and np.array_equal(np.lexsort(t.T[::-1]), np.arange(len(t)))


# (the fixed-size workloads cfg2/cfg3/cfg5 take minutes to hours on the executor; the 1 M-particle cfg2 ran once by hand)
@pytest.mark.parametrize("extra", [[], ["--levelset-variant", "1", "--no-cpu-baseline"], ["--levelset-variant", "0", "--no-cpu-baseline"]], ids=["default", "levelset_variant_1", "levelset_variant_0"])
def test_bench_single_rank_on_executor(oracle_mod, extra, tmp_path):
    cmd = [sys.executable, LAUNCHER, "bench.py", "--particles", "12000", "--steps", "2", "--warmup", "1", "--cpu-sample-particles", "8000",
           "--dump-outputs", str(tmp_path / "dump")] + extra
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, SS_EMUL_THREADS="4"))
    assert r.returncode == 0, r.stderr[-3000:]
    d = _check_line(r.stdout, 1, 2)
    _check_dump(str(tmp_path / "dump"), d)
    assert d["config"]["plan_settling_steps"] == 0                      # a single GPU has no plan to settle
    if "--no-cpu-baseline" not in extra:
        assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    want = int(extra[extra.index("--levelset-variant") + 1]) if "--levelset-variant" in extra else 2
    assert d["config"]["levelset_variant"] == want and d["roofline"]["launches_per_step"] >= (2 if want else 1)
    # the extra end-to-end reading of a single-GPU run: the documented front-end call on a pageable numpy array
    assert d["e2e_frontend"]["value"] > 0


@pytest.mark.parametrize("protocol", ["stats", "two_call", "callback"])
def test_bench_two_ranks_on_executor(oracle_mod, protocol, tmp_path):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), LAUNCHER, "bench.py", "--gpus", "2", "--particles", "12000", "--steps", "2",
           "--warmup", "1", "--runner-protocol", protocol, "--dump-outputs", str(tmp_path / "dump")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, SS_EMUL_THREADS="3", OMP_NUM_THREADS="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    d = _check_line(r.stdout, 2, 2)
    _check_dump(str(tmp_path / "dump"), d)
    assert d["config"]["parallelism"].endswith("x2") and d["mesh"]["vertices"] > 0
    # warm-up 1 < the runner's exploration frames: the bench ran untimed settling steps (the same number on both ranks, or the
    # collectives inside a step would have dead-locked) and says so
    assert 1 <= d["config"]["plan_settling_steps"] <= 9


def test_bench_reference_arm_contract(oracle_mod):
    """`bench.py --impl reference` (the reference wheel on the host cores): one JSON line with the arm's own metric / config keys, the
    `cpu_baseline` describing this run and an `e2e` that repeats the line's value with no host<->device traffic."""
    if not oracle_mod.reference_available():
        pytest.skip("oracle/_ref not unpacked")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--particles", "20000", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    assert d["unit"] == "Mparticles/s" and d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 2 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["bounded_sample"] is False and "workload" in d["config"]


def test_bench_reference_arm_under_torchrun_prints_once(oracle_mod):
    """Launched like the scaling run (N ranks): rank 0 alone runs the reference and prints; the other ranks exit 0 without work."""
    if not oracle_mod.reference_available():
        pytest.skip("oracle/_ref not unpacked")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(free_port()),
           os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--particles", "20000", "--steps", "1", "--warmup", "0"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["impl"] == "reference" and json.loads(lines[0])["n_gpus"] == 2
