"""GPU parity of the PCG loop through every SpMV kernel the plan can select, against the CPU oracle ref_pcg.

The loop does not just call y = A x.  Every iteration launches the SpMV instantiation with the fused dot epilogue, whose
per-tile partials of p.q give alpha = rho / (p.q), and, depending on the plan, the split-row fix-up (k_spmv_fixup) and the
first level of a two-level p.q sum (k_stage_reduce, more than 8192 partials).  A dot that drops one tile's partial, reads a
stale x entry or counts a split row's head twice leaves y correct and the iteration count within its slack: only the
solution drifts.  So every case here
  * asserts plan_info(), so that a plan that quietly falls back to another kernel fails instead of passing;
  * runs one iteration from x0 = 0: x_1 = (rho_0 / p_0.A p_0) z_0 carries the relative error of the fused dot as it is,
    and is pinned to 1e-12 (a missing tile partial moves alpha by far more);
  * solves to tol 1e-13 and compares flag, iteration count, residual history and solution with the oracle.
Tolerance names and values are those of test_gpu_pcg.py.  ref_pcg is pinned to the unmodified reference by the golden tests.
"""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import ref_pcg as R

pytestmark = pytest.mark.gpu

X_RTOL = 1e-10        # solution parity at tol 1e-13
ITER_SLACK = 2        # iteration counts may differ by +-1-2 across summation orders
RESVEC_RTOL = 1e-9    # residual history, first RESVEC_HEAD entries
RESVEC_HEAD = 12
STEP_RTOL = 1e-12     # one iteration: x_1 and RelRes carry the rounding of rho_0 and p_0.q_0 only
STEP_TOL = 1e-12      # tolerance of the one-iteration solve (never reached by a system of order > 1)
TOL = 1e-13
MAXITER = 5000


# ------------------------------------------------------------------------------------------------------ systems
def _arrowhead(k=10, m=3):
    """poisson27(k) + I bordered by m dense rows and columns: rows of k^3 + m entries that no 256-item tile holds (split-row
    plan).  Border entries are at most 0.1 in magnitude, so every interior row keeps a diagonal margin > 0.7; each border
    diagonal exceeds its row's absolute sum by at least 1: symmetric and strictly diagonally dominant, hence SPD."""
    rng = np.random.default_rng(0)
    n0 = k ** 3
    B = rng.uniform(0.05, 0.1, size=(n0, m)) * rng.choice([-1.0, 1.0], size=(n0, m))
    C = np.full((m, m), 0.05)
    np.fill_diagonal(C, 0.0)
    np.fill_diagonal(C, np.abs(B).sum(axis=0) + np.abs(C).sum(axis=1) + 1.0 + np.arange(m))
    A = sp.bmat([[R.poisson27(k) + sp.identity(n0), sp.csr_matrix(B)], [sp.csr_matrix(B.T), sp.csr_matrix(C)]]).tocsr()
    A.sort_indices()
    return A


def _tiny(n):
    """Dense SPD G G^T + n I of order n (n = 3: one 3x3 node block)."""
    G = np.random.default_rng(100 + n).standard_normal((n, n))
    K = G @ G.T + n * np.eye(n)
    return sp.csr_matrix(0.5 * (K + K.T))


@functools.lru_cache(maxsize=None)
def _ebe_subdomain():
    """Synthetic pattern groups (as test_gpu_assemble's mixed-pattern case) with SPD Ke = G G^T + nd I: sizes 3 .. 96, sign
    flips, clamped dofs, element counts that are no multiple of 8 or 128, one empty group.  Nine distinct non-empty 24-dof
    Ke plus the empty 24-dof group need ten constant-memory slots, of which there are 8: whatever other operators hold, at
    least two non-empty 24-dof groups run on k_ebe_warp next to the k_ebe_t24 ones."""
    from pcg_mpi_solver_b200.partition import SubdomainData, TypeGroup
    rng = np.random.default_rng(21)
    ndof = 603
    groups = []

    def spd(nd):
        G = rng.standard_normal((nd, nd))
        K = G @ G.T + nd * np.eye(nd)
        return 0.5 * (K + K.T)

    def add(loc, ke):
        nd, ne = loc.shape
        groups.append(TypeGroup(len(groups), loc.astype(np.int64), rng.random((nd, ne)) < 0.2, rng.random(ne) + 0.5, ke, np.arange(ne)))

    def scattered(nd, ne):
        return np.stack([rng.choice(ndof, nd, replace=False) for _ in range(ne)], axis=1) if ne else np.zeros((nd, 0))

    add(scattered(24, 0), spd(24))                                   # empty group (takes a slot all the same)
    add(np.arange(ndof).reshape(-1, 3).T, spd(3))                    # 201 elements cover every dof: K is positive definite
    for nd, ne in [(12, 37), (33, 19), (60, 11), (96, 5)]:
        add(scattered(nd, ne), spd(nd))
    for ne in (13, 27, 41, 55, 69, 83, 97, 111, 131):                # nine distinct 24-dof pattern matrices
        add(scattered(24, ne), spd(24))
    eff = np.sort(rng.choice(ndof, 540, replace=False))              # 63 clamped dofs
    return SubdomainData(0, 1, np.arange(ndof), np.arange(ndof // 3), eff, groups, [], [], [], np.ones(ndof), np.zeros(ndof),
                         np.zeros(ndof), eff.size, ndof)


def _ebe_assembled():
    from pcg_mpi_solver_b200.partition import _assemble
    sub = _ebe_subdomain()
    K = _assemble(sub.groups, sub.ndof)
    return K[sub.loc_dof_eff][:, sub.loc_dof_eff].tocsr()


MATRICES = {
    "hex": lambda: R.hex_box_csr((9, 7, 5), (0, 0, 0), (9, 7, 5)),
    "poisson": lambda: R.poisson27(12),
    "hex_clamped": lambda: R.hex_box_csr((14, 12, 10), (0, 0, 0), (14, 12, 10)),
    "hex_interior": lambda: R.hex_box_csr((8, 6, 4), (4, 0, 2), (4, 3, 2)),   # no clamped face: singular, b = A x* is consistent
    "arrow": _arrowhead,
    "poisson48": lambda: R.poisson27(48),
    "ebe": _ebe_assembled,
    **{f"tiny{n}": functools.partial(_tiny, n) for n in (1, 2, 3, 4, 7)},
}


@functools.lru_cache(maxsize=None)
def _system(name):
    A = MATRICES[name]()
    A.sort_indices()
    b = A @ np.random.default_rng(1).standard_normal(A.shape[0])
    return A, b, 1.0 / A.diagonal()


@functools.lru_cache(maxsize=None)
def _oracle(name, precond, tol, maxiter):
    """ref_pcg on the scipy matrix in fp64, cached per (matrix, preconditioner, tol, maxiter) for the whole module."""
    A, b, minv = _system(name)
    hist = []
    ref = R.ref_pcg([R.CsrPart(A, b)], [minv], tol, maxiter, exist_dp0=precond, resvec=hist)
    ref["resvec"] = np.array(hist)
    return ref


# ------------------------------------------------------------------------------------------------------ checks
def _csr_operator(cuda, monkeypatch, name, env, expect, index64=False):
    """Sets the plan's environment BEFORE the matrix is created (the plan reads it then) and asserts the plan it produced."""
    from pcg_mpi_solver_b200.csr import CsrMatrix
    from pcg_mpi_solver_b200.solver import SubdomainOperator
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    M = CsrMatrix.from_scipy(_system(name)[0], device=cuda, index64=index64)
    info = M.plan_info()
    print(f"plan of {name} (index64={index64}):", " ".join(f"{k}={info[k]}" for k in ("ntiles", "snap", "split_rows", "staged", "tma",
                                                                                       "lanes", "index_mode")))
    for k, v in expect.items():
        assert info[k] == v, (k, v, info)
    return SubdomainOperator(M), info


def _check_first_step(op, name, precond=True):
    from pcg_mpi_solver_b200 import solve
    _, b, minv = _system(name)
    ref = _oracle(name, precond, STEP_TOL, 1)
    x, flag, relres, iters = solve(op, b, minv if precond else None, STEP_TOL, 1)
    assert flag == ref["Flag"]
    # while XMin is still bound to X (no improvement recorded) Iter hangs on a rounding-level comparison
    assert iters == ref["Iter"] or (ref["aliased"] and iters == 1)
    X = ref["X"][0]
    assert np.linalg.norm(x - X) <= STEP_RTOL * np.linalg.norm(X), np.linalg.norm(x - X) / np.linalg.norm(X)
    if flag == 0:   # a system of order one is solved by the first step: both residuals are rounding noise
        assert relres <= STEP_TOL and ref["RelRes"] <= STEP_TOL
    else:
        assert abs(relres - ref["RelRes"]) <= STEP_RTOL * ref["RelRes"], (relres, ref["RelRes"])


def _check_full_solve(op, name, precond=True, **kw):
    from pcg_mpi_solver_b200 import solve
    _, b, minv = _system(name)
    ref = _oracle(name, precond, TOL, MAXITER)
    x, flag, relres, iters, info = solve(op, b, minv if precond else None, TOL, MAXITER, record_resvec=True, return_info=True, **kw)
    assert flag == ref["Flag"], (flag, ref["Flag"])
    assert abs(iters - ref["Iter"]) <= ITER_SLACK, (iters, ref["Iter"])
    if flag == 0:
        assert relres <= TOL
    hist = ref["resvec"]
    m = min(RESVEC_HEAD, len(hist), len(info.resvec))
    keep = hist[:m] > 1e-5 * hist[0]      # only the tiny systems reach rounding level within RESVEC_HEAD iterations
    np.testing.assert_allclose(info.resvec[:m][keep], hist[:m][keep], rtol=RESVEC_RTOL)
    X = ref["X"][0]
    assert np.linalg.norm(x - X) <= X_RTOL * np.linalg.norm(X), np.linalg.norm(x - X) / np.linalg.norm(X)
    return x, flag, relres, iters, info.resvec


# ------------------------------------------------------------------------------------------------------ 1-3: every kernel
SNAPPED = {"snap": 1, "split_rows": 0}
VARIANTS = {
    **{f"merge_ldg_lanes{l}": ({"PCGB_SPMV_TMA": "0", "PCGB_SPMV_LANES": str(l)},
                               {"staged": 0, "tma": 0, "lanes": l, "index_mode": 0}) for l in (4, 8, 16, 32)},
    "merge_tma": ({"PCGB_SPMV_TMA": "1", "PCGB_SPMV_STAGE": "0"}, {"staged": 0, "tma": 1, "index_mode": 0}),
    "staged": ({"PCGB_SPMV_STAGE": "1", "PCGB_SPMV_PERSIST": "0"}, {"staged": 1, "tma": 1, "index_mode": 0}),
    "persist": ({"PCGB_SPMV_BSR": "0", "PCGB_SPMV_T3": "0"}, {"staged": 2, "tma": 1, "index_mode": 0}),
    **{f"persist_t3_lanes{l}": ({"PCGB_SPMV_BSR": "0", "PCGB_SPMV_T3": "1", "PCGB_SPMV_LANES3": str(l)},
                                {"staged": 2, "tma": 1, "index_mode": 1, "lanes": l}) for l in (4, 32)},
    **{f"bsr_cw{cw}_uni{uni}_inplace{ip}": ({"PCGB_BSR_MIN_UNIFORM_PCT": "0", "PCGB_BSR_CW": str(cw), "PCGB_BSR_UNI": str(uni),
                                             "PCGB_BSR_INPLACE": str(ip)}, {"staged": 2, "tma": 1, "index_mode": 2})
       for cw in (6, 8, 12) for uni in (0, 1) for ip in (0, 1)},
}


def _matrices_of(variant):
    if variant.startswith("persist_t3"):
        return ("hex",)                                       # column triples: 3 dofs per node
    if variant.startswith("bsr"):
        return ("hex", "hex_clamped", "hex_interior")         # node blocks
    return ("hex", "poisson")


CASES = [(v, m) for v in VARIANTS for m in _matrices_of(v)]


def _table_operator(cuda, monkeypatch, variant, matrix, index64=False):
    env, expect = VARIANTS[variant]
    op, info = _csr_operator(cuda, monkeypatch, matrix, env, {**SNAPPED, **expect}, index64)
    assert info["ntiles"] >= 2, info     # several tiles, so that every partial of p.q counts
    return op, info


@pytest.mark.parametrize("variant,matrix", CASES)
def test_first_step_pins_fused_dot(cuda, monkeypatch, variant, matrix):
    op, _ = _table_operator(cuda, monkeypatch, variant, matrix)
    _check_first_step(op, matrix)


@pytest.mark.parametrize("variant,matrix", CASES)
def test_full_solve_matches_oracle(cuda, monkeypatch, variant, matrix):
    op, _ = _table_operator(cuda, monkeypatch, variant, matrix)
    _check_full_solve(op, matrix)


# ------------------------------------------------------------------------------------------------------ 4: split rows
SPLIT_VARIANTS = {
    "merge_ldg": ({"PCGB_SPMV_TMA": "0"}, {"staged": 0, "tma": 0}),
    "merge_tma": ({"PCGB_SPMV_STAGE": "0"}, {"staged": 0, "tma": 1}),
    "staged": ({"PCGB_SPMV_STAGE": "1", "PCGB_SPMV_PERSIST": "0"}, {"staged": 1, "tma": 1}),
    "persist": ({}, {"staged": 2, "tma": 1, "index_mode": 0}),
}


def _split_operator(cuda, monkeypatch, variant, index64=False):
    env, expect = SPLIT_VARIANTS[variant]
    op, info = _csr_operator(cuda, monkeypatch, "arrow", {"PCGB_SPMV_TILE": "256", **env}, {"snap": 0, **expect}, index64)
    # the border rows span several tiles: their heads go to carry[] and k_spmv_fixup adds them inside the loop
    assert info["split_rows"] >= 3 and info["ntiles"] > 100, info
    return op, info


@pytest.mark.parametrize("variant", SPLIT_VARIANTS)
def test_split_rows_first_step(cuda, monkeypatch, variant):
    op, _ = _split_operator(cuda, monkeypatch, variant)
    _check_first_step(op, "arrow")


@pytest.mark.parametrize("variant", SPLIT_VARIANTS)
def test_split_rows_full_solve(cuda, monkeypatch, variant):
    op, _ = _split_operator(cuda, monkeypatch, variant)
    _check_full_solve(op, "arrow")


@pytest.mark.parametrize("variant", SPLIT_VARIANTS)
def test_split_rows_graph_and_batching_are_exact(cuda, monkeypatch, variant):
    """k_spmv_fixup captured in the CUDA graph and replayed in batches gives the same bits as direct launches polled every
    iteration."""
    from pcg_mpi_solver_b200 import solve
    op, _ = _split_operator(cuda, monkeypatch, variant)
    _, b, minv = _system("arrow")
    base = solve(op, b, minv, TOL, MAXITER, check_every=1, use_graph=False, record_resvec=True, return_info=True)
    for use_graph in (False, True):
        for check_every in (1, 5):
            got = solve(op, b, minv, TOL, MAXITER, check_every=check_every, use_graph=use_graph, record_resvec=True, return_info=True)
            assert got[1:4] == base[1:4], (use_graph, check_every)
            assert np.array_equal(got[0], base[0]) and np.array_equal(got[4].resvec, base[4].resvec), (use_graph, check_every)


# ------------------------------------------------------------------------------------------------------ 3: offset width
@pytest.mark.parametrize("variant,matrix", CASES + [(f"split_{v}", "arrow") for v in SPLIT_VARIANTS])
def test_int64_offsets_are_bit_identical(cuda, monkeypatch, variant, matrix):
    """The int64 row-offset instantiations (the C5 production path) run the same plan as int32: same bits in the loop."""
    from pcg_mpi_solver_b200 import solve
    _, b, minv = _system(matrix)
    out = []
    for index64 in (False, True):
        if variant.startswith("split_"):
            op, info = _split_operator(cuda, monkeypatch, variant[len("split_"):], index64)
        else:
            op, info = _table_operator(cuda, monkeypatch, variant, matrix, index64)
        x, flag, relres, iters, si = solve(op, b, minv, TOL, MAXITER, record_resvec=True, return_info=True)
        out.append((info, x, (flag, relres, iters), si.resvec))
    (i32, x32, s32, h32), (i64, x64, s64, h64) = out
    assert i32 == i64
    assert s32 == s64 and np.array_equal(x32, x64) and np.array_equal(h32, h64)


# ------------------------------------------------------------------------------------------------------ 5: > 8192 tiles
# poisson27(48): 110592 rows + 2863288 non-zeros = 2973880 merge items
MANY_TILES = {
    "merge_tma_tile256": ({"PCGB_SPMV_TILE": "256", "PCGB_SPMV_PERSIST": "0", "PCGB_SPMV_STAGE": "0"}, {"staged": 0, "tma": 1}),
    "staged_tile256": ({"PCGB_SPMV_TILE": "256", "PCGB_SPMV_PERSIST": "0", "PCGB_SPMV_STAGE": "1"}, {"staged": 1, "tma": 1}),
    # 8193 tiles: the last block of k_stage_reduce (4096 partials per block) holds a single partial
    "merge_tma_tile363": ({"PCGB_SPMV_TILE": "363", "PCGB_SPMV_PERSIST": "0", "PCGB_SPMV_STAGE": "0"}, {"staged": 0, "tma": 1}),
}


def _many_tiles_operator(cuda, monkeypatch, variant):
    env, expect = MANY_TILES[variant]
    op, info = _csr_operator(cuda, monkeypatch, "poisson48", env, {**SNAPPED, **expect})
    assert info["ntiles"] > 8192, info    # more partials than one reduction pass takes: two-level sum
    if variant.endswith("tile363"):
        assert 1 <= info["ntiles"] % 4096 <= 3, info
    return op


@pytest.mark.parametrize("variant", MANY_TILES)
def test_many_tiles_first_step(cuda, monkeypatch, variant):
    _check_first_step(_many_tiles_operator(cuda, monkeypatch, variant), "poisson48")


@pytest.mark.parametrize("variant", MANY_TILES)
def test_many_tiles_full_solve(cuda, monkeypatch, variant):
    _check_full_solve(_many_tiles_operator(cuda, monkeypatch, variant), "poisson48")


# ------------------------------------------------------------------------------------------------------ 6: tiny systems
TINY_VARIANTS = {
    "default": ({}, {"staged": 2, "tma": 1, "index_mode": 0}),
    "merge_ldg": ({"PCGB_SPMV_TMA": "0"}, {"staged": 0, "tma": 0, "index_mode": 0}),
    "bsr": ({"PCGB_BSR_MIN_UNIFORM_PCT": "0"}, {"staged": 2, "tma": 1, "index_mode": 2}),
}
TINY_CASES = [(v, n) for n in (1, 2, 3, 4, 7) for v in TINY_VARIANTS if v != "bsr" or n == 3]


@pytest.mark.parametrize("precond", [True, False], ids=["jacobi", "none"])
@pytest.mark.parametrize("variant,n", TINY_CASES)
def test_tiny_systems(cuda, monkeypatch, variant, n, precond):
    env, expect = TINY_VARIANTS[variant]
    op, info = _csr_operator(cuda, monkeypatch, f"tiny{n}", env, {**SNAPPED, **expect, "ntiles": 1})
    _check_first_step(op, f"tiny{n}", precond)
    _check_full_solve(op, f"tiny{n}", precond)


# ------------------------------------------------------------------------------------------------------ 7: matrix-free
def test_ebe_operator_in_the_loop(cuda):
    """EbeMatrix (k_ebe_t24 + k_ebe_warp, fp64 atomics) per entry against the host assembly, then inside the PCG loop."""
    import torch
    sub = _ebe_subdomain()
    A, _, _ = _system("ebe")
    op = sub.to_operator(device=cuda, kind="ebe")
    assert sum(1 for g in sub.groups if g.ke.shape[0] == 24 and g.loc_dof.shape[1] > 0) == 9
    for seed in range(3):
        x = np.random.default_rng(seed).standard_normal(A.shape[0])
        y = op.A.apply_local(torch.from_numpy(x).to(cuda)).cpu().numpy()
        err = np.abs(y - A @ x) / (abs(A) @ np.abs(x))
        assert err.max() <= 1e-13, err.max()
    np.testing.assert_allclose(op.jacobi().cpu().numpy(), 1.0 / A.diagonal(), rtol=1e-13)
    _check_first_step(op, "ebe")
    _check_full_solve(op, "ebe")
