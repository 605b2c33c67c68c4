"""Pin the CPU oracle (oracle/ref_pcg.py) and the product's subdomain builder to the UNMODIFIED reference.

Golden vectors in tests/golden/ were produced by running /root/reference under the fake-MPI shim
(oracle/make_golden_hex.py, make_golden_concrete.py, make_golden_probe.py):
  hex_ref.{json,npz}        structured hex model in the reference's MDF format, 1/2/4/8 parts + METIS 4:
                            Flag, Iter, RelRes and the FULL solution vector of every run
  concrete_ref*.{json,npz}  data/concrete.zip, 1 and 8 parts: Flag, Iter, RelRes, ||U||, sampled U, neighbour table
  concrete_probe.*          outputs of the reference's own calcMPFint / updatePreconditioner / updateBC
"""
import json
import os

import numpy as np
import pytest

from oracle import ref_pcg as R
from oracle.hex_mdf import write_hex_mdf

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _concrete_zip():
    p = os.path.join(ROOT, "oracle", "_ref", "concrete.zip")
    if not os.path.exists(p):
        pytest.skip("data/concrete.zip not staged (__graft_entry__.build() stages it where the reference checkout is readable)")
    return p


@pytest.fixture(scope="module")
def hex_gold():
    with open(os.path.join(GOLD, "hex_ref.json")) as f:
        meta = json.load(f)
    return meta, np.load(os.path.join(GOLD, "hex_ref.npz"))


@pytest.fixture(scope="module")
def hex_model(hex_gold, tmp_path_factory):
    from pcg_mpi_solver_b200.model import load_mdf
    path = tmp_path_factory.mktemp("hexmdf")
    write_hex_mdf(str(path), tuple(hex_gold[0]["ng"]))
    return load_mdf(str(path), name="hexmodel")


def _gather(subs, xs, ndof):
    u = np.zeros(ndof)
    for s, x in zip(subs, xs):
        u[s.dof_eff_global] = x
    return u


@pytest.mark.parametrize("case", ["box1", "box2", "box4", "box8", "metis4"])
def test_oracle_ebe_reproduces_reference_hex(hex_gold, hex_model, case):
    """Restated element-by-element PCG == the reference, same iteration count, solution to rounding."""
    from pcg_mpi_solver_b200.partition import build_subdomains
    meta, arr = hex_gold
    run = meta["runs"][case]
    ep = arr[f"elepart_{case}"].astype(np.int64) if run["nparts"] > 1 else np.zeros(hex_model.n_elem, dtype=np.int64)
    subs = build_subdomains(hex_model, ep, run["nparts"], assemble=False)
    # builder parity with the reference builder's tables
    for s, tab in zip(subs, run["parts"]):
        assert s.nbr == tab["nbr"] and [len(v) for v in s.ovrlp_full] == tab["n_ovrlp"]
        assert s.ndof == tab["ndof"] and s.weights_full.sum() == tab["wsum"]
    parts = [R.EbePart(s.to_refmeshpart()) for s in subs]
    R.update_bc(parts)
    op = R.Operator(parts)
    out = R.ref_pcg(parts, op.jacobi(), meta["tol"], meta["maxiter"], nglob=hex_model.n_dof_eff)
    assert out["Flag"] == run["Flag"] == 0
    assert out["Iter"] == run["Iter"]
    assert abs(out["RelRes"] - run["RelRes"]) <= 1e-6 * run["RelRes"]
    u = _gather(subs, out["X"], hex_model.n_dof)
    uref = arr[f"U_{case}"]
    assert np.linalg.norm(u - uref) <= 1e-12 * np.linalg.norm(uref)


@pytest.mark.parametrize("case", ["box1", "box4", "metis4"])
def test_oracle_csr_and_builder_assembly_hex(hex_gold, hex_model, case):
    """The assembled-CSR form (what the CUDA path consumes) gives the reference's answer."""
    from pcg_mpi_solver_b200.partition import build_subdomains
    meta, arr = hex_gold
    run = meta["runs"][case]
    ep = arr[f"elepart_{case}"].astype(np.int64) if run["nparts"] > 1 else np.zeros(hex_model.n_elem, dtype=np.int64)
    subs = build_subdomains(hex_model, ep, run["nparts"], assemble=True)
    parts = [R.CsrPart(s.A, s.b, s.nbr, s.ovrlp, s.weights, part_id=s.id) for s in subs]
    op = R.Operator(parts)
    out = R.ref_pcg(parts, op.jacobi(), meta["tol"], meta["maxiter"], nglob=hex_model.n_dof_eff)
    assert out["Flag"] == 0 and abs(out["Iter"] - run["Iter"]) <= 1
    u = _gather(subs, out["X"], hex_model.n_dof)
    uref = arr[f"U_{case}"]
    assert np.linalg.norm(u - uref) <= 1e-10 * np.linalg.norm(uref)
    if run["nparts"] == 1:  # the box generator of the oracle agrees with the general assembly
        ng = tuple(meta["ng"])
        B = R.hex_box_csr(ng, (0, 0, 0), ng, h=1.0 / ng[0])
        assert abs(B - subs[0].A).max() <= 1e-14 * abs(B).max()


def test_concrete_operator_probe_matches_reference():
    """calcMPFint / updatePreconditioner / updateBC of the reference itself vs the restatement on the
    product builder's data (1 part)."""
    from pcg_mpi_solver_b200.partition import partition_mesh
    with open(os.path.join(GOLD, "concrete_probe.json")) as f:
        g = json.load(f)
    arr = np.load(os.path.join(GOLD, "concrete_probe.npz"))
    sub = partition_mesh(_concrete_zip(), 1, assemble=False)[0]
    assert sub.ndof == g["ndof"] and sub.n == g["neff"]
    part = R.EbePart(sub.to_refmeshpart())
    dofv = sub.dof_vector
    v = np.sin(0.001 * dofv) + 0.25 * np.cos(0.37 * dofv)
    fixed = np.setdiff1d(np.arange(sub.ndof), sub.loc_dof_eff)
    v[fixed] = 0.0
    y = part.matvec_full(v)
    assert abs(np.linalg.norm(y) - g["norm_y"]) <= 1e-13 * g["norm_y"]
    np.testing.assert_allclose(y[arr["idx"]], arr["y"], rtol=1e-12, atol=1e-9 * np.abs(arr["y"]).max())
    minv = R.Operator([part]).jacobi()[0]
    np.testing.assert_allclose(minv[::101], arr["minv"], rtol=1e-13)
    R.update_bc([part])
    fext = np.zeros(sub.ndof)
    fext[sub.loc_dof_eff] = part.b
    np.testing.assert_allclose(fext[arr["idx"]][np.isin(arr["idx"], sub.loc_dof_eff)],
                               arr["fext"][np.isin(arr["idx"], sub.loc_dof_eff)], rtol=1e-13, atol=1e-300)


def test_concrete_builder_tables_match_reference():
    """8-way partition of concrete: neighbour table, shared-dof counts and weight sums of the reference
    builder (golden G5 / make_golden_concrete.py)."""
    from pcg_mpi_solver_b200.partition import partition_mesh
    with open(os.path.join(GOLD, "concrete_ref.json")) as f:
        g = json.load(f)
    ep = np.load(os.path.join(GOLD, "concrete_elepart_8.npy")).astype(np.int64)
    subs = partition_mesh(_concrete_zip(), 8, elepart=ep, assemble=False)
    tabs = g["runs"]["8"]["parts"]
    for s in subs:
        t = tabs[str(s.id)]
        assert s.nbr == t["nbrs"] and [len(v) for v in s.ovrlp_full] == t["shared_dofs"]
        assert s.ndof == t["NDOF"] and s.n == t["NDofEff"]
        assert s.weights_full.sum() == t["weight_sum"] and s.weights.sum() == t["weight_sum_eff"]
    assert sum(s.weights_full.sum() for s in subs) == g["GlobNDof"]
    assert sum(s.weights.sum() for s in subs) == g["GlobNDofEff"]


def test_metis_partition_is_usable():
    """METIS_PartMeshDual through the CUDA-toolkit libmetis: balanced 8-way split of concrete (the reference
    calls mgmetis with the same routine, run_metis.py:88; partition parity itself is unpinned - see DESIGN.md)."""
    from pcg_mpi_solver_b200.metis import run_metis
    from pcg_mpi_solver_b200.model import load_mdf
    m = load_mdf(_concrete_zip())
    ep = run_metis(m.node_flat, m.node_offset, 8)
    counts = np.bincount(ep, minlength=8)
    assert counts.sum() == m.n_elem and counts.min() > 0.9 * m.n_elem / 8 and counts.max() < 1.1 * m.n_elem / 8
    gold = np.load(os.path.join(GOLD, "concrete_elepart_8.npy"))
    assert np.array_equal(ep, gold)  # deterministic for a given METIS build


@pytest.mark.slow
@pytest.mark.skipif(os.environ.get("PCGB_SLOW") != "1", reason="~4 min: full concrete solves with the numpy oracle (PCGB_SLOW=1)")
@pytest.mark.parametrize("nparts", [1, 8])
def test_oracle_reproduces_reference_concrete(nparts):
    from pcg_mpi_solver_b200.partition import partition_mesh
    with open(os.path.join(GOLD, "concrete_ref.json")) as f:
        g = json.load(f)
    run = g["runs"][str(nparts)]
    ep = np.load(os.path.join(GOLD, "concrete_elepart_8.npy")).astype(np.int64) if nparts == 8 else None
    subs = partition_mesh(_concrete_zip(), nparts, elepart=ep, assemble=False)
    from threadpoolctl import threadpool_limits
    parts = [R.EbePart(s.to_refmeshpart()) for s in subs]
    with threadpool_limits(limits=1):  # the reference pins BLAS to one thread (pcg_solver.py:10-15): same summation order
        R.update_bc(parts)
        op = R.Operator(parts)
        out = R.ref_pcg(parts, op.jacobi(), g["Tol"], g["MaxIter"], nglob=g["GlobNDofEff"])
    assert out["Flag"] == run["Flag"] == 0 and abs(out["Iter"] - run["Iter"]) <= 1
    if out["Iter"] == run["Iter"]:
        assert abs(out["RelRes"] - run["RelRes"]) <= 1e-2 * run["RelRes"]
    u = _gather(subs, out["X"], g["GlobNDof"])
    assert abs(np.linalg.norm(u) - run["norm2_U"]) <= 1e-12 * run["norm2_U"]
    s = np.load(os.path.join(GOLD, "concrete_ref_samples.npz"))
    np.testing.assert_allclose(u[s["idx"]], s[f"U{nparts}"], rtol=0, atol=1e-10 * np.abs(s[f"U{nparts}"]).max())


@pytest.mark.parametrize("case,nparts", [("maxiter3", 1), ("maxiter30", 1), ("maxiter3", 4)])
def test_oracle_maxiter_exit_matches_reference(hex_model, case, nparts):
    """Non-converged exit (pcg_solver.py:566-598) against the UNMODIFIED reference (oracle/make_golden_maxiter.py): the
    reference binds MP_XMin = MP_X and updates X in place (:379-380, :516), so before the first recorded improvement the
    exported solution is the LATEST iterate (maxiter3: residual still growing), afterwards the frozen minimum."""
    from pcg_mpi_solver_b200.hexmesh import block_grid, partition_blocks
    from pcg_mpi_solver_b200.partition import build_subdomains
    with open(os.path.join(GOLD, "hex_maxiter_ref.json")) as f:
        meta = json.load(f)
    arr = np.load(os.path.join(GOLD, "hex_maxiter_ref.npz"))
    run = meta["runs"][case]
    ng = tuple(meta["ng"])
    ep = np.zeros(hex_model.n_elem, dtype=np.int64)
    if nparts > 1:     # the exit path does not depend on the partition: same golden for a 4-box split
        nx, ny, nz = ng
        for r, b in enumerate(partition_blocks(ng, block_grid(nparts))):
            ez, ey, ex = np.meshgrid(np.arange(b.e0[2], b.e0[2] + b.ne[2]), np.arange(b.e0[1], b.e0[1] + b.ne[1]),
                                     np.arange(b.e0[0], b.e0[0] + b.ne[0]), indexing="ij")
            ep[((ez * ny + ey) * nx + ex).ravel()] = r
    subs = build_subdomains(hex_model, ep, nparts, assemble=False)
    parts = [R.EbePart(s.to_refmeshpart()) for s in subs]
    R.update_bc(parts)
    out = R.ref_pcg(parts, R.Operator(parts).jacobi(), meta["tol"], run["maxiter"], nglob=hex_model.n_dof_eff)
    assert out["Flag"] == run["Flag"] == 1
    # Iter is decided by `NormR < NormR_Act` between the true and the recurrence residual of the SAME iterate when XMin is
    # still aliased (a rounding-level comparison): either branch is the reference's behaviour; the solution is the same
    assert out["Iter"] in ((run["Iter"], 1) if case == "maxiter3" else (run["Iter"],))
    assert abs(out["RelRes"] - run["RelRes"]) <= 1e-9 * run["RelRes"]
    u = _gather(subs, out["X"], hex_model.n_dof)
    uref = arr[f"U_{case}"]
    assert np.linalg.norm(u - uref) <= 1e-12 * np.linalg.norm(uref)
