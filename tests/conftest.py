import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")


def free_port() -> int:
    """A currently unused TCP port on 127.0.0.1 for torchrun rendezvous in multi-process tests."""
    import socket
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def load_npz_parts(name):
    """Arrays of tests/golden/<name>.npz and of its continuation files <name>_1.npz, <name>_2.npz, ... (fixtures are split so that
    no file exceeds 1 MB)."""
    d, i, path = {}, 0, os.path.join(GOLDEN, name + ".npz")
    while os.path.exists(path):
        z = np.load(path, allow_pickle=False)
        d.update({k: z[k] for k in z.files})
        i += 1
        path = os.path.join(GOLDEN, f"{name}_{i}.npz")
    return d


def load_golden(name):
    d = load_npz_parts(name)
    if "kwargs" in d:
        d["kwargs"] = json.loads(str(d["kwargs"]))
    return d


@pytest.fixture(scope="session")
def oracle_mod():
    import oracle
    oracle.build()
    return oracle


@pytest.fixture(scope="session")
def ss():
    """The product package with its CUDA library built and loaded (no compute without a GPU)."""
    import splashsurf_b200
    from splashsurf_b200 import build
    build.build()
    splashsurf_b200.load_library()
    if os.environ.get("SS_TEST_EMULATED"):
        # developer switch (never set by the driver): run GPU-marked tests on the CPU executor of the CUDA sources, e.g.
        #   SS_TEST_EMULATED=1 pytest tests -m gpu -k "not full_size and not dam_ and not multi_gpu and not global_big"
        import ctypes
        from test_emulated_pipeline import build_emulated_library
        splashsurf_b200._LIB = splashsurf_b200._bind(ctypes.CDLL(build_emulated_library()))
    return splashsurf_b200


def digest(*parts) -> str:
    """sha256 over byte strings and arrays (dtype, shape and contents): a reference output stored by its digest still pins every bit."""
    import hashlib
    h = hashlib.sha256()
    for p in parts:
        if not isinstance(p, (bytes, bytearray)):
            a = np.ascontiguousarray(p)
            h.update(f"{a.dtype.str}{a.shape}".encode())
            p = a.tobytes()
        h.update(p)
    return h.hexdigest()


REFERENCE_OUTPUTS = os.path.join(GOLDEN, "reference_outputs.json")


@pytest.fixture(scope="session")
def reference_output():
    """Outputs of the reference binary that tests compare against, stored in tests/golden/reference_outputs.json (digests, names,
    flags).  `reference_output(key, run)` returns the stored value; with SS_RECORD_REFERENCE=1 it calls `run()` (which runs the
    reference in oracle/_ref) instead.  At the end of such a session the values recorded are merged into the file: keys of tests
    that did not run keep their stored values, and a value is the reference's output whether or not the test then passed.  The
    keys of GPU-marked tests are recorded by a `-m gpu` session, on a GPU or on the CPU executor (SS_TEST_EMULATED=1):
        SS_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"
        SS_RECORD_REFERENCE=1 SS_TEST_EMULATED=1 python -m pytest tests -m gpu -k "reference_datasets or gpu_postprocess"
    """
    stored = json.load(open(REFERENCE_OUTPUTS)) if os.path.exists(REFERENCE_OUTPUTS) else {}
    if not os.environ.get("SS_RECORD_REFERENCE"):
        def get(key, run):
            assert key in stored, f"{key} is missing from {REFERENCE_OUTPUTS}: record it with SS_RECORD_REFERENCE=1"
            return stored[key]
        yield get
        return

    def record(key, run):
        stored[key] = run()
        return stored[key]
    yield record
    with open(REFERENCE_OUTPUTS, "w") as f:
        json.dump(dict(sorted(stored.items())), f, indent=0)
        f.write("\n")


MESH_CASES = ["cfg1_ref", "cube16_ref", "cube16_scalar_ref", "splash_small_ref", "splash_aabb_ref", "global_cube_ref",
              "global_autodisable_ref"]
