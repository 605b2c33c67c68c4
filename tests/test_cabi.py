"""CPU checks of the C ABI: the library loads without a GPU, exports every symbol include/pcgb200.h
declares, and refuses to compute without a device (no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "pcgb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pcgb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from pcg_mpi_solver_b200 import _lib
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/pcgb200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(names)
    assert lib.pcgb_version() == 200


def test_struct_layouts_match_header():
    from pcg_mpi_solver_b200 import _lib
    sizes = (ctypes.c_int32 * 4)()
    _lib.load().pcgb_abi_sizes(sizes)                      # sizeof() as the C++ compiler sees the structs of pcgb200.h
    assert ctypes.sizeof(_lib.Options) == sizes[0]
    assert ctypes.sizeof(_lib.Result) == sizes[1]
    assert ctypes.sizeof(_lib.HexBox) == sizes[2] == 36
    assert ctypes.sizeof(_lib.EbeGroup) == sizes[3]


def test_operator_refuses_foreign_matrix_handles(monkeypatch):
    """SubdomainOperator hands A.handle to the library as a pcgb_csr_t or a pcgb_ebe_t.  Anything else - an
    EbeMatrixColored holds a pcgb_ebe2_t - is refused with TypeError before any call into the library."""
    import torch
    from pcg_mpi_solver_b200 import _lib
    from pcg_mpi_solver_b200.ebe import EbeMatrixColored
    from pcg_mpi_solver_b200.solver import SubdomainOperator

    def no_library(*args, **kwargs):
        raise AssertionError("the library was called")

    monkeypatch.setattr(_lib, "load", no_library)
    colored = EbeMatrixColored.__new__(EbeMatrixColored)    # a handle-carrying object of the wrong kind, no device needed
    colored.shape, colored.device, colored._h = (6, 6), torch.device("cpu"), ctypes.c_void_p()
    for A in (colored, object()):
        with pytest.raises(TypeError, match="CsrMatrix or an EbeMatrix"):
            SubdomainOperator(A)


def test_no_cpu_fallback():
    import numpy as np
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pcg_mpi_solver_b200 import _lib, solve
    from oracle import ref_pcg as R
    lib = _lib.load()
    assert lib.pcgb_device_count() == 0
    h = ctypes.c_void_p()
    rc = lib.pcgb_csr_create(1, 1, 0, 8, 0, None, None, None, ctypes.byref(h))
    assert rc == -4 and b"no CPU fallback" in lib.pcgb_last_error()
    A = R.poisson27(4)
    with pytest.raises(_lib.PcgbError):
        solve(A, np.ones(A.shape[0]), None, 1e-8, 10)


def test_product_does_not_import_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    pkg = os.path.join(ROOT, "pcg_mpi_solver_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), (dirpath, f)


def test_bench_reference_arm_schema():
    """`bench.py --impl reference` prints ONE JSON line with the contract keys (small mesh so it runs in seconds).  The CPU arm
    times the difference of a 1+K and a 1 iteration run: at 16^3 and K = 3 that is ~4 ms, below the host's scheduling noise,
    and the value can come out negative; at 32^3 and K = 20 it is ~0.1 s."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--block", "32", "--steps", "20", "--cpu-iters", "20"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"].startswith("subdomain-iterations/s") and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_bench_parity_checker_and_goldens():
    """bench.py's parity block: the committed oracle goldens exist for every GPU count of the default workload, an exact history
    passes, a perturbed one fails (the bench then exits with code 3), a missing golden is reported as such."""
    import importlib.util
    import json

    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for n in (1, 2, 4, 8):
        gold, path = bench.golden_resvec(128, n)
        assert gold is not None and len(gold["resvec"]) == 41 and gold["n_gpus"] == n, path
        res = bench.resvec_parity(np.array(gold["resvec"][:21]), gold["normb"], gold, path)
        assert res["ok"] is True and res["max_rel_err"] == 0.0 and res["checked_iterations"] == 10
        bad = np.array(gold["resvec"][:21])
        bad[7] *= 1 + 1e-7
        assert bench.resvec_parity(bad, gold["normb"], gold, path)["ok"] is False
        assert bench.resvec_parity(np.array(gold["resvec"][:21]), gold["normb"] * (1 + 1e-6), gold, path)["ok"] is False
    gold, path = bench.golden_resvec(96, 3)
    assert gold is None and bench.resvec_parity(np.ones(5), 1.0, gold, path)["ok"] is None
    # the 1e8-dof goldens of the north-star size (160^3 per GPU at 8 GPUs = 320^3 elements)
    g160, _ = bench.golden_resvec(160, 8)
    assert g160 is not None and g160["n_global"] == 3 * 320 * 321 * 321


def test_c_demo_compiles_links_and_refuses_to_run_without_a_gpu(tmp_path, build_c_demo):
    """The boundary is a C ABI: a plain-C caller compiles and links against the header and the shared object; without a device it
    fails loudly (exit code 4) instead of falling back to anything."""
    import subprocess

    import torch
    exe = build_c_demo(str(tmp_path / "cabi_demo"))
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_gpu_cabi_demo.py runs it")
    r = subprocess.run([exe, "8"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 4 and "no CPU fallback" in r.stdout


def test_resvec_goldens_are_partition_independent():
    """Two goldens describe the SAME global problem cut differently: 256^3 elements as one 256^3 block (8 oracle processes on one
    'GPU' mesh) and as 2x2x2 blocks of 128^3 (the N=8 bench mesh).  The reference's PCG is partition-independent up to round-off
    (SURVEY 8(c) G6), so the two residual histories must agree far below the bench's 1e-9 gate."""
    import json

    import numpy as np
    gold = os.path.join(ROOT, "tests", "golden")
    a = json.load(open(os.path.join(gold, "hex128_N8_resvec.json")))
    b = json.load(open(os.path.join(gold, "hex256_N1_resvec.json")))
    assert a["ng"] == b["ng"] == [256, 256, 256] and a["n_global"] == b["n_global"]
    ra, rb = np.array(a["resvec"]), np.array(b["resvec"])
    assert abs(a["normb"] - b["normb"]) <= 1e-14 * a["normb"]
    assert np.abs(ra - rb).max() / ra.max() <= 1e-11
