"""Matrix-free EBE operator (SURVEY 8(f1)): the reference's own operator form on the GPU, against the assembled
CSR path, the CPU oracle and the reference's golden iteration count on concrete.  First run on a B200 at the very
end of round 1 (both tests green); not yet profiled or tuned - opt-in via to_operator(kind="ebe")."""
import os

import numpy as np
import pytest

from oracle import ref_pcg as R
from oracle.hex_mdf import write_hex_mdf

pytestmark = pytest.mark.gpu


def test_ebe_operator_matches_csr_and_oracle_hex(cuda, tmp_path):
    import torch
    from pcg_mpi_solver_b200.model import load_mdf
    from pcg_mpi_solver_b200.partition import partition_mesh
    write_hex_mdf(str(tmp_path), (9, 7, 5))
    sub = partition_mesh(load_mdf(str(tmp_path)), 1, assemble=True)[0]
    op = sub.to_operator(device=cuda, kind="ebe")
    x = np.random.default_rng(0).standard_normal(sub.n)
    y = op.apply(torch.from_numpy(x).to(cuda)).cpu().numpy()
    yref = sub.A @ x
    assert np.abs(y - yref).max() <= 1e-12 * (abs(sub.A) @ np.abs(x)).max()
    np.testing.assert_allclose(op.jacobi().cpu().numpy(), 1.0 / sub.A.diagonal(), rtol=1e-13)
    b = torch.from_numpy(sub.b).to(cuda)
    xs, info = op.solve(b, op.jacobi(), 1e-10, 5000)
    ref = R.ref_pcg([R.CsrPart(sub.A, sub.b)], [1.0 / sub.A.diagonal()], 1e-10, 5000)
    assert info.flag == ref["Flag"] == 0 and abs(info.iters - ref["Iter"]) <= 2
    # the solution itself: near tol 1e-10 one CG iteration more or less moves x by ~1e-12 relative on this mesh
    X = ref["X"][0]
    assert np.linalg.norm(xs.cpu().numpy() - X) <= 1e-10 * np.linalg.norm(X)


def test_ebe_operator_concrete(cuda):
    import torch
    from pcg_mpi_solver_b200.partition import partition_mesh
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    zp = os.path.join(root, "oracle", "_ref", "concrete.zip")
    if not os.path.exists(zp):
        pytest.skip("concrete.zip not staged")
    sub = partition_mesh(zp, 1, assemble=False)[0]
    ebe = sub.to_operator(device=cuda, kind="ebe")
    csr = sub.to_operator(device=cuda, kind="csr")
    x = torch.randn(sub.n, dtype=torch.float64, device=cuda)
    ye, yc = ebe.apply(x), csr.apply(x)
    assert float((ye - yc).abs().max() / yc.abs().max()) <= 1e-12
    xs, info = ebe.solve(torch.from_numpy(sub.b).to(cuda), ebe.jacobi(), 1e-7, 10000)
    assert info.flag == 0 and abs(info.iters - 1085) <= 2


def test_two_live_ebe_operators_keep_their_own_pattern_matrices(cuda):
    """The constant-memory slots of the 24-dof pattern matrices are shared per device: creating a second operator with a
    DIFFERENT Ke must not disturb a live first one (slots are content-deduplicated and reference-counted)."""
    import torch
    from pcg_mpi_solver_b200.ebe import EbeMatrix
    from pcg_mpi_solver_b200.hexmesh import HexBlock, generate_matrix, hex_type_group
    ops, refs = [], []
    for nu in (0.3, 0.1, 0.3, 0.45):                       # third one shares the first one's slot
        blk = HexBlock((6, 5, 4), (0, 0, 0), (6, 5, 4), h=0.25, nu=nu)
        grp, eff, ndof = hex_type_group(blk)
        ops.append(EbeMatrix([grp], eff, ndof, device=cuda))
        refs.append(generate_matrix(blk, device=cuda))
    x = torch.randn(ops[0].shape[0], dtype=torch.float64, device=cuda)
    for rounds in range(2):                                 # interleaved applications, all operators alive
        for E, A in zip(ops, refs):
            ye, yc = E.apply_local(x), A.spmv(x)
            assert float((ye - yc).abs().max() / yc.abs().max()) <= 1e-12
    del ops[1]                                               # releasing one operator leaves the others intact
    blk = HexBlock((6, 5, 4), (0, 0, 0), (6, 5, 4), h=0.25, nu=0.2)
    grp, eff, ndof = hex_type_group(blk)
    extra = EbeMatrix([grp], eff, ndof, device=cuda)         # may reuse the freed slot
    for E, A in zip(ops + [extra], [refs[0], refs[2], refs[3], generate_matrix(blk, device=cuda)]):
        ye, yc = E.apply_local(x), A.spmv(x)
        assert float((ye - yc).abs().max() / yc.abs().max()) <= 1e-12
