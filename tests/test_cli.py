"""The file-format-compatible solver stage (pcg_mpi_solver_b200/pcg_solver.py, SURVEY 8(f3)/(f4)): reads the
reference's fixtures / settings files and writes result files the reference's readers understand."""
import json
import os
import pickle
import zlib

import numpy as np
import pytest

from oracle import ref_pcg as R
from oracle import run_reference as rr
from oracle.cli_workdir import FRAME_CASES, same_fixture, setup_workdir

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _unpack_reference_files(prefix, dst):
    """Writes the files that the unmodified reference produced under `prefix` of tests/golden/cli_ref.npz
    (oracle/make_golden_cli.py) into the directory `dst`."""
    os.makedirs(dst, exist_ok=True)
    with np.load(os.path.join(GOLD, "cli_ref.npz")) as z:
        for key in z.files:
            if key.startswith(prefix + "/") and "/" not in key[len(prefix) + 1:]:
                z[key].tofile(os.path.join(dst, key[len(prefix) + 1:]))


def _oracle_backend(mp, ranks):
    """CPU checker standing in for the GPU so that the file formats can be exercised without a device."""
    from pcg_mpi_solver_b200.pcg_solver import _default_backend  # noqa: F401  (signature reference)
    from pcg_mpi_solver_b200.partition import SubdomainData, TypeGroup
    part = R.EbePart(mp)
    eff = part.eff
    groups = [TypeGroup(int(g["ElemTypeId"]), g["ElemList_LocDofVector"], g["ElemList_SignVector"], g["ElemList_Ck"], g["ElemStiffMat"], None)
              for g in mp["SubDomainData"]["StrucDataList"]]
    sub = SubdomainData(int(mp["Id"]), 1, np.asarray(mp["DofVector"]), np.asarray(mp["NodeIdVector"]), eff, groups, [], [], [],
                        np.asarray(mp["DofWeightVector"], dtype=float), np.asarray(mp["RefLoadVector"], dtype=float),
                        np.asarray(mp["Ud"], dtype=float), int(mp["GlobData"]["GlobNDofEff"]), int(mp["GlobData"]["GlobNDof"]))
    minv = R.Operator([part]).jacobi()

    def solve_step(b, x0, tol, maxiter):
        part.b, part.x0 = b, x0
        out = R.ref_pcg([part], minv, tol, maxiter, nglob=sub.n_global_eff)
        return out["X"][0], out["Flag"], out["RelRes"], out["Iter"]

    return sub, solve_step


def test_cli_file_formats_roundtrip_cpu(tmp_path):
    """export_mesh_parts -> run() -> the reference's result readers; solution equals the reference's golden run."""
    from pcg_mpi_solver_b200.model import load_mdf
    from pcg_mpi_solver_b200.partition import partition_mesh
    from pcg_mpi_solver_b200.pcg_solver import export_mesh_parts, read_mesh_part, run
    with open(os.path.join(GOLD, "hex_ref.json")) as f:
        meta = json.load(f)
    gold = np.load(os.path.join(GOLD, "hex_ref.npz"))
    ng = tuple(meta["ng"])
    work, mdf, info = setup_workdir(tmp_path, ng, meta["tol"], meta["maxiter"])
    subs = partition_mesh(load_mdf(mdf, "hexmodel"), 1, assemble=False)
    prefix = os.path.join(work, "data", "ModelData", "MPI") + "/"
    export_mesh_parts(prefix, subs)
    mp = read_mesh_part(prefix, 1, 0)
    assert np.array_equal(mp["LocDofEff"], subs[0].loc_dof_eff) and mp["NDOF"] == subs[0].ndof
    out = run(1, 0, workdir=work, backend=_oracle_backend, quiet=True)
    res, u = rr.read_results(work, "hexmodel", 1, 1, info["ndof"])     # reads like file_operations.py:517-531 / export_vtk.py:157-159
    run1 = meta["runs"]["box1"]
    assert res["Flag"] == run1["Flag"] == 0 and res["Iter"] == run1["Iter"]
    assert np.linalg.norm(u - gold["U_box1"]) <= 1e-12 * np.linalg.norm(gold["U_box1"])
    vec = os.path.join(work, "data", "Results_Run1", "ResVecData")
    for name in ("Dof", "NodeId", "U_0", "U_1"):
        assert os.path.exists(os.path.join(vec, name + ".mpidat")) and os.path.exists(os.path.join(vec, name + "_metadat.npy"))
    assert list(np.load(os.path.join(vec, "Time_T.npy"))) == [0.0, 0.0]
    td = np.load(os.path.join(work, "data", "Results_Run1", "PlotData", "hexmodel_MP1_TimeData.npz"), allow_pickle=True)["TimeData"].item()
    assert {"TotalTime", "Mean_CalcTime", "Mean_CommWaitTime", "Mean_FileReadTime", "Flag", "Iter", "RelRes"} <= set(td)


def test_cli_multi_step_ramp_cpu(tmp_path):
    """Time-step shell (pcg_solver.py:1002-1008): a two-step load ramp reuses A and M; the solution scales with delta."""
    from pcg_mpi_solver_b200.model import load_mdf
    from pcg_mpi_solver_b200.partition import partition_mesh
    from pcg_mpi_solver_b200.pcg_solver import export_mesh_parts, run
    work, mdf, info = setup_workdir(tmp_path, (4, 3, 3), 1e-11, 2000, deltas=(0, 0.5, 1.0))
    subs = partition_mesh(load_mdf(mdf, "hexmodel"), 1, assemble=False)
    export_mesh_parts(os.path.join(work, "data", "ModelData", "MPI") + "/", subs)
    out = run(7, 0, workdir=work, backend=_oracle_backend, quiet=True)
    assert list(out["Flag"]) == [0, 0, 0] and out["Iter"][1] > 0
    _, u1 = rr.read_results(work, "hexmodel", 1, 7, info["ndof"], frame=1)
    _, u2 = rr.read_results(work, "hexmodel", 1, 7, info["ndof"], frame=2)
    assert np.linalg.norm(u2 - 2.0 * u1) <= 1e-8 * np.linalg.norm(u2)   # linear problem: delta 1.0 vs 0.5


def test_cli_reads_the_reference_builders_fixture_cpu(tmp_path):
    """The fixture written by the UNMODIFIED reference builder is consumed as is."""
    from pcg_mpi_solver_b200.pcg_solver import run
    work, mdf, info = setup_workdir(tmp_path, (5, 4, 3), 1e-10, 3000)
    # the reference's run_metis.py + partition_mesh.py on this model -> 1_metadat.npy, 1_0.mpidat
    _unpack_reference_files("fixture_543", os.path.join(work, "data", "ModelData", "MPI"))
    out = run(3, 0, workdir=work, backend=_oracle_backend, quiet=True)
    assert out["Flag"][1] == 0
    A = R.hex_box_csr((5, 4, 3), (0, 0, 0), (5, 4, 3), h=info["h"])
    x = out["Un"][out["sub"].loc_dof_eff]
    b = info["F"][info["eff"]]
    assert np.linalg.norm(b - A @ x) <= 1e-10 * np.linalg.norm(b) * (1 + 1e-6)


@pytest.mark.parametrize("rate,frms", FRAME_CASES)
def test_cli_export_frames_match_the_reference(tmp_path, rate, frms):
    """ExportFrms is a NESTED, 1-BASED list (np.array(ExportFrms, int)[0] - 1, pcg_solver.py:156-159) and the step-0 frame is
    written only when the ExportNow predicate holds for step 0 (:854-859): same set of U_k files, same contents, same Time_T
    as the unmodified reference run on the same fixture (its result files: tests/golden/cli_ref.npz)."""
    from pcg_mpi_solver_b200.pcg_solver import run
    work, mdf, info = setup_workdir(tmp_path, (4, 3, 3), 1e-11, 2000)
    _unpack_reference_files("fixture_433", os.path.join(work, "data", "ModelData", "MPI"))
    settings = {"TimeHistoryParam": {"ExportFlag": True, "ExportFrmRate": rate, "ExportFrms": frms, "PlotFlag": False,
                                     "TimeStepDelta": [0, 0.25, 0.5, 1.0], "ExportVars": "U"}, "SolverParam": {"Tol": 1e-11, "MaxIter": 2000}}
    with open(os.path.join(work, "__pycache__", "GlobSettings.zpkl"), "wb") as f:
        f.write(zlib.compress(pickle.dumps(settings, pickle.HIGHEST_PROTOCOL)))
    ref_dir = os.path.join(work, "reference_ResVecData")                 # the unmodified reference's run on this fixture
    _unpack_reference_files(f"frames{FRAME_CASES.index((rate, frms))}", ref_dir)
    run(2, 0, workdir=work, backend=_oracle_backend, quiet=True)         # the file-compatible stage
    our_dir = os.path.join(work, "data", "Results_Run2", "ResVecData")
    ref_files = sorted(f for f in os.listdir(ref_dir) if f.endswith(".mpidat"))
    assert sorted(f for f in os.listdir(our_dir) if f.endswith(".mpidat")) == ref_files
    for f in ref_files:
        a, b = np.fromfile(os.path.join(ref_dir, f), dtype=np.uint8), np.fromfile(os.path.join(our_dir, f), dtype=np.uint8)
        if f.startswith("U_"):
            ua, ub = a.view(np.float64), b.view(np.float64)
            assert ua.shape == ub.shape and np.linalg.norm(ua - ub) <= 1e-9 * max(np.linalg.norm(ua), 1e-300)
        else:
            assert np.array_equal(a, b)
    if os.path.exists(os.path.join(ref_dir, "Time_T.npy")):
        assert list(np.load(os.path.join(ref_dir, "Time_T.npy"))) == list(np.load(os.path.join(our_dir, "Time_T.npy")))
    else:
        assert not os.path.exists(os.path.join(our_dir, "Time_T.npy"))


@pytest.mark.gpu
def test_cli_on_gpu_matches_reference_golden(cuda, tmp_path):
    """Same pipeline with the CUDA backend (device assembly + pcgb_solve) against the reference's golden run."""
    from pcg_mpi_solver_b200.model import load_mdf
    from pcg_mpi_solver_b200.partition import partition_mesh
    from pcg_mpi_solver_b200.pcg_solver import export_mesh_parts, run
    with open(os.path.join(GOLD, "hex_ref.json")) as f:
        meta = json.load(f)
    gold = np.load(os.path.join(GOLD, "hex_ref.npz"))
    ng = tuple(meta["ng"])
    work, mdf, info = setup_workdir(tmp_path, ng, meta["tol"], meta["maxiter"])
    subs = partition_mesh(load_mdf(mdf, "hexmodel"), 1, assemble=False)
    export_mesh_parts(os.path.join(work, "data", "ModelData", "MPI") + "/", subs)
    run(1, 0, workdir=work, quiet=True)
    res, u = rr.read_results(work, "hexmodel", 1, 1, info["ndof"])
    run1 = meta["runs"]["box1"]
    assert res["Flag"] == 0 and abs(res["Iter"] - run1["Iter"]) <= 2 and res["RelRes"] <= meta["tol"]
    assert np.linalg.norm(u - gold["U_box1"]) <= 1e-8 * np.linalg.norm(gold["U_box1"])


@pytest.mark.parametrize("nparts", [1, 2])
def test_reference_solver_consumes_the_product_builders_fixture(tmp_path, nparts):
    """Drop-in the other way round: the UNMODIFIED reference solver (pcg_solver.py under the fake-MPI shim) ran on the
    fixture written by the product's partition_mesh()/export_mesh_parts() and reproduced its own golden run
    (oracle/make_golden_cli.py stored that fixture and the reference's result): the builder still writes that fixture."""
    from pcg_mpi_solver_b200.model import load_mdf
    from pcg_mpi_solver_b200.partition import partition_mesh
    from pcg_mpi_solver_b200.pcg_solver import export_mesh_parts, read_mesh_part
    with open(os.path.join(GOLD, "hex_ref.json")) as f:
        meta = json.load(f)
    gold = np.load(os.path.join(GOLD, "hex_ref.npz"))
    ng = tuple(meta["ng"])
    work, mdf, info = setup_workdir(tmp_path, ng, meta["tol"], meta["maxiter"])
    case = "box1" if nparts == 1 else "box2"
    ep = gold[f"elepart_{case}"].astype(np.int64) if nparts > 1 else None
    subs = partition_mesh(load_mdf(mdf, "hexmodel"), nparts, elepart=ep, assemble=False)
    prefix = os.path.join(work, "data", "ModelData", "MPI") + "/"
    export_mesh_parts(prefix, subs)
    ref_prefix = os.path.join(work, "consumed_by_reference") + "/"
    _unpack_reference_files(f"consumes{nparts}/fixture", ref_prefix)
    for p in range(nparts):
        assert same_fixture(read_mesh_part(prefix, nparts, p), read_mesh_part(ref_prefix, nparts, p)), p
    # the reference's run (pcg_solver.py, one process per part) on that fixture, as recorded: these asserts compare two
    # golden files (cli_ref.npz and hex_ref.npz) and compute nothing; they keep a regenerated cli_ref.npz honest
    with np.load(os.path.join(GOLD, "cli_ref.npz")) as z:
        flag, iters, u = int(z[f"consumes{nparts}/Flag"]), int(z[f"consumes{nparts}/Iter"]), z[f"consumes{nparts}/U"]
    run = meta["runs"][case]
    assert flag == 0 and iters == run["Iter"]
    assert np.linalg.norm(u - gold[f"U_{case}"]) <= 1e-12 * np.linalg.norm(gold[f"U_{case}"])
