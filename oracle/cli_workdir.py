"""Work directories of the file-format drop-in tests (tests/test_cli.py) and of the script that records the reference's
side of them (oracle/make_golden_cli.py)."""
import os

import numpy as np

from oracle import run_reference as rr
from oracle.hex_mdf import write_hex_mdf

FRAME_CASES = [(0, [[2, 3]]), (2, [[2]]), (0, [])]       # (ExportFrmRate, ExportFrms) of the frame-export test


def setup_workdir(path, ng, tol, maxiter, deltas=(0, 1)):
    """A work directory laid out like read_input_model.py leaves it (read_input_model.py:24-48)."""
    from pcg_mpi_solver_b200.pcg_solver import exportz
    work = str(path)
    mdf = os.path.join(work, "data", "ModelData", "MDF") + "/"
    info = write_hex_mdf(mdf, ng)
    os.makedirs(os.path.join(work, "__pycache__"), exist_ok=True)
    os.makedirs(os.path.join(work, "data", "ModelData", "MPI"), exist_ok=True)   # read_input_model.py:31-36
    exportz(os.path.join(work, "__pycache__", "ModelDataPaths.zpkl"),
            {"ScratchPath": os.path.join(work, "data"), "MDF_Path": mdf, "PyDataPath_Part": os.path.join(work, "data", "ModelData", "MPI") + "/",
             "ModelName": "hexmodel"})
    rr.write_settings(work, tol, maxiter, deltas)
    return work, mdf, info


def same_fixture(a, b):
    """Structural equality of two decoded fixtures (dicts / lists / arrays / scalars), arrays compared exactly."""
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(same_fixture(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return isinstance(b, (list, tuple)) and len(a) == len(b) and all(same_fixture(x, y) for x, y in zip(a, b))
    if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        return np.asarray(a).dtype == np.asarray(b).dtype and np.array_equal(a, b)
    return type(a) is type(b) and a == b
