#!/usr/bin/env python
"""Golden files for the drop-in tests of tests/test_cli.py, produced by the UNMODIFIED reference.

Those tests check file-format compatibility in both directions: the product's solver stage reads the fixture the
reference's builder writes, writes the same result files as the reference's solver, and the reference's solver reads
the fixture the product's builder writes.  This script runs the reference stages once and stores, byte for byte, every
file those tests take from it, so that the tests run without the reference:
    fixture_543/, fixture_433/    the reference builder's fixture (1 part) of the 5x4x3 and 4x3x3 hex models
    frames<k>/                    the reference solver's ResVecData files for the k-th ExportFrms case of the test
    consumes<N>/fixture/          the product builder's fixture (N parts) of the hex_ref model that the reference ran on
    consumes<N>/U                 the reference solver's solution on that fixture (Flag, Iter beside it)
Writes tests/golden/cli_ref.npz (relative path -> uint8 bytes; scalars as 0-d arrays).  Needs the reference."""
import json
import os
import pickle
import shutil
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import run_reference as rr  # noqa: E402
from oracle.cli_workdir import FRAME_CASES, same_fixture, setup_workdir  # noqa: E402

work = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix="pcgb_ref_cli_")
shutil.rmtree(work, ignore_errors=True)
os.makedirs(work)
out = {}


def grab(prefix, directory, names=None):
    for f in sorted(os.listdir(directory)):
        if (names is None or f in names) and os.path.isfile(os.path.join(directory, f)):
            out[f"{prefix}/{f}"] = np.fromfile(os.path.join(directory, f), dtype=np.uint8)


def mpi_dir(w):
    return os.path.join(w, "data", "ModelData", "MPI")


# the reference builder's fixtures
for ng, tol, maxiter in (((5, 4, 3), 1e-10, 3000), ((4, 3, 3), 1e-11, 2000)):
    tag = "fixture_" + "".join(map(str, ng))
    w = os.path.join(work, tag)
    setup_workdir(w, ng, tol, maxiter)
    rr.metis_stage(w, 1)
    rr.partition_stage(w, 1)
    grab(tag, mpi_dir(w))

# the reference solver's exported frames, one case of test_cli_export_frames_match_the_reference each
for k, (rate, frms) in enumerate(FRAME_CASES):
    w = os.path.join(work, f"frames{k}")
    setup_workdir(w, (4, 3, 3), 1e-11, 2000)
    rr.metis_stage(w, 1)
    rr.partition_stage(w, 1)
    # the test hands fixture_433 to the product's solver in place of this one: the same but for the work-directory
    # paths in GlobData, which the solver stage takes from __pycache__/ModelDataPaths.zpkl instead
    mine, first = rr.load_mesh_part(w, 1, 0), rr.load_mesh_part(os.path.join(work, "fixture_433"), 1, 0)
    for m in (mine, first):
        for key in ("ScratchPath", "MDF_Path", "PyDataPath_Part"):
            m["GlobData"].pop(key)
    assert same_fixture(mine, first)
    settings = {"TimeHistoryParam": {"ExportFlag": True, "ExportFrmRate": rate, "ExportFrms": frms, "PlotFlag": False,
                                     "TimeStepDelta": [0, 0.25, 0.5, 1.0], "ExportVars": "U"}, "SolverParam": {"Tol": 1e-11, "MaxIter": 2000}}
    with open(os.path.join(w, "__pycache__", "GlobSettings.zpkl"), "wb") as f:
        f.write(zlib.compress(pickle.dumps(settings, pickle.HIGHEST_PROTOCOL)))
    rr.solve_stage(w, 1, run_id=1)
    ref_dir = os.path.join(w, "data", "Results_Run1", "ResVecData")
    grab(f"frames{k}", ref_dir, [f for f in os.listdir(ref_dir) if f.endswith(".mpidat")] + ["Time_T.npy"])

# the reference solver on the product builder's fixture
from pcg_mpi_solver_b200.model import load_mdf  # noqa: E402
from pcg_mpi_solver_b200.partition import partition_mesh  # noqa: E402
from pcg_mpi_solver_b200.pcg_solver import export_mesh_parts  # noqa: E402

with open(os.path.join(ROOT, "tests", "golden", "hex_ref.json")) as f:
    meta = json.load(f)
gold = np.load(os.path.join(ROOT, "tests", "golden", "hex_ref.npz"))
for nparts, case in ((1, "box1"), (2, "box2")):
    w = os.path.join(work, f"consumes{nparts}")
    _, mdf, info = setup_workdir(w, tuple(meta["ng"]), meta["tol"], meta["maxiter"])
    ep = gold[f"elepart_{case}"].astype(np.int64) if nparts > 1 else None
    subs = partition_mesh(load_mdf(mdf, "hexmodel"), nparts, elepart=ep, assemble=False)
    export_mesh_parts(mpi_dir(w) + "/", subs)
    grab(f"consumes{nparts}/fixture", mpi_dir(w))
    rr.solve_stage(w, nparts, run_id=5)
    res, u = rr.read_results(w, "hexmodel", nparts, 5, info["ndof"])
    out[f"consumes{nparts}/U"] = u
    out[f"consumes{nparts}/Flag"] = np.array(res["Flag"])
    out[f"consumes{nparts}/Iter"] = np.array(res["Iter"])
    print(f"consumes{nparts}: Flag {res['Flag']} Iter {res['Iter']}")

dst = os.path.join(ROOT, "tests", "golden", "cli_ref.npz")
np.savez_compressed(dst, **out)
print(f"wrote {dst}: {len(out)} entries, {os.path.getsize(dst)} bytes")
