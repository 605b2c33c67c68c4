"""Python host side of the PCG hot path: `solve(A, b, M, tol, maxiter)` and the operator handle.

Reference surface being replaced (SURVEY.md 8(b)):
    PCG(RefMeshPart)                     pcg_solver.py:356-598   -> solve() / SubdomainOperator.solve()
    calcMPFint(x_full, RefMeshPart)      pcg_solver.py:339-342   -> SubdomainOperator.apply()
    updatePreconditioner(RefMeshPart)    pcg_solver.py:346-352   -> SubdomainOperator.jacobi()
    MPI_SUM(v, GlobData)                 pcg_solver.py:622-628   -> Communicator.allreduce_sum()

Mapping of solve()'s arguments onto the reference's per-rank state:
    A        K[Eff,Eff] of this rank (CsrMatrix / SubdomainOperator with its halo plan)
    b        Fext[LocDofEff]
    M        InvDiagPreCondVector0 (the INVERSE diagonal, applied as z = M*r, :447); None = identity
             (ExistDP0 False, :451); the string "jacobi" builds it from A like updatePreconditioner
    tol      GlobData['Tol']        maxiter  GlobData['MaxIter']
    x0       Un[LocDofEff]          w        DofWeightVector_Eff (taken from the operator if omitted)
Return value (x, flag, relres, iters) follows MATLAB pcg like the reference: flag 0 converged,
1 maxiter, 2 preconditioner produced inf, 3 stagnation, 4 breakdown; iters = Iter after the +1 (:584).

All arithmetic runs in libpcgb200.so (CUDA, sm_100a); torch only owns the device buffers.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .csr import CsrMatrix
from .ebe import EbeMatrix


def _allgather_bytes(blob: bytes, group=None):
    """All-gather of one bytes object per rank over the torch.distributed side channel (rank order)."""
    import torch.distributed as dist
    box = [None] * dist.get_world_size(group)
    dist.all_gather_object(box, blob, group=group)
    return box


class Communicator:
    """Communicator of the solver ranks (one rank = one GPU = one subdomain, pcg_solver.py:91; replaces COMM_WORLD).

    Data path (see include/pcgb200.h): `transport == "peer"` = the library's own kernels over CUDA-IPC mapped peer memory
    (NVLink / NVSwitch; all-reduce fused into the reduction kernel, halo values stored straight into the neighbours'
    buffers), `"nccl"` = ncclAllReduce / ncclSend / ncclRecv.  The host side channel (torch.distributed) only carries the
    NCCL unique id and the IPC handles."""

    def __init__(self, rank: int, nranks: int, unique_id: bytes | None, device=None, allgather=None):
        self.rank, self.nranks = rank, nranks
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._h = ctypes.c_void_p()
        self._allgather = allgather
        self.peer_error = None
        self._has_nccl = unique_id is not None
        uid = (ctypes.c_ubyte * _lib.UNIQUE_ID_BYTES).from_buffer_copy(unique_id) if unique_id is not None else None
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().pcgb_comm_create(rank, nranks, uid, ctypes.byref(self._h)), "pcgb_comm_create")
        if allgather is not None and nranks > 1:
            self.exchange_windows(allgather)

    def exchange_windows(self, allgather) -> bool:
        """Export this rank's window, all-gather the handles, import the peers' windows.  On failure (no CUDA IPC in this
        environment) the communicator stays on NCCL; the reason is kept in `peer_error`."""
        lib = _lib.load()
        self._allgather = allgather
        self.peer_error = None
        blob = (ctypes.c_ubyte * _lib.IPC_BLOB_BYTES)()
        ok = True
        with torch.cuda.device(self.device):
            if lib.pcgb_comm_window_export(self._h, blob) != 0:
                ok, self.peer_error = False, lib.pcgb_last_error().decode()
        blobs = allgather(bytes(blob) if ok else b"")
        if not all(len(b) == _lib.IPC_BLOB_BYTES for b in blobs):
            return False                                   # some rank could not export: everybody stays on NCCL
        buf = (ctypes.c_ubyte * (_lib.IPC_BLOB_BYTES * self.nranks)).from_buffer_copy(b"".join(blobs))
        with torch.cuda.device(self.device):
            rc = lib.pcgb_comm_window_import(self._h, buf)
        if rc != 0:
            self.peer_error = lib.pcgb_last_error().decode()
        oks = allgather(b"1" if rc == 0 else b"0")
        if not all(o == b"1" for o in oks):
            if self.transport == "peer":                   # imported here but not everywhere: do not use it
                lib.pcgb_comm_set_transport(self._h, _lib.TRANSPORT_NCCL)
            return False
        return True

    @staticmethod
    def unique_id() -> bytes:
        uid = (ctypes.c_ubyte * _lib.UNIQUE_ID_BYTES)()
        _lib.check(_lib.load().pcgb_comm_unique_id(uid), "pcgb_comm_unique_id")
        return bytes(uid)

    @classmethod
    def from_torch_distributed(cls, device=None, nccl: bool = True, group=None):
        """Bootstrap from an initialised torch.distributed group: rank 0 creates the NCCL unique id and broadcasts it,
        then the peer windows are exchanged (side channel only; the data path uses the library's own communicator).
        nccl=False builds a peer-only communicator (e.g. several ranks sharing one GPU in a test)."""
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        uid = None
        if nccl:
            box = [cls.unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0, group=group)
            uid = box[0]
        return cls(rank, world, uid, device, allgather=lambda b: _allgather_bytes(b, group))

    @property
    def handle(self):
        return self._h

    @property
    def transport(self) -> str:
        return "peer" if _lib.load().pcgb_comm_transport(self._h) == _lib.TRANSPORT_PEER else "nccl"

    def set_transport(self, name: str) -> None:
        _lib.check(_lib.load().pcgb_comm_set_transport(self._h, _lib.TRANSPORT_PEER if name == "peer" else _lib.TRANSPORT_NCCL),
                   "pcgb_comm_set_transport")

    def allreduce_sum(self, t: torch.Tensor) -> torch.Tensor:
        assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().pcgb_allreduce_sum(self._h, _lib.ptr(t), t.numel(), _lib.stream_ptr()), "pcgb_allreduce_sum")
        return t

    def __del__(self):
        try:
            if self._h:
                _lib.load().pcgb_comm_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass


@dataclass
class SolveInfo:
    flag: int = 1
    iters: int = 0
    relres: float = 0.0
    normb: float = 0.0
    imin: int = 0
    stag: int = 0
    moresteps: int = 0
    too_small_tol: bool = False
    matvecs: int = 0
    launches: int = 0
    loop_ms: float = 0.0
    spmv_ms: float = 0.0
    spmv_timed: int = 0
    loop_iters: int = 0
    setup_ms: float = 0.0
    final_ms: float = 0.0
    phase_ms: dict | None = None
    resvec: np.ndarray | None = None


class SubdomainOperator:
    """K[Eff,Eff] of one subdomain + its interface-exchange plan: the `A` of solve().

    nbr_ranks / ovrlp are NbrMPIdVector / OvrlpLocalDofVecList of the reference restricted to free dofs
    and renumbered in the Eff numbering (partition.py does that); weights is DofWeightVector_Eff.
    With comm=None (one subdomain) it is just the matrix.
    """

    def __init__(self, A, comm: Communicator | None = None, nbr_ranks=(), ovrlp=(), weights=None,
                 n_global: int | None = None):
        # the C side reads A.handle as a pcgb_csr_t or a pcgb_ebe_t: any other handle (EbeMatrixColored holds a
        # pcgb_ebe2_t) would be misread as one of them, so it is refused before anything reaches the library
        if not isinstance(A, (CsrMatrix, EbeMatrix)):
            raise TypeError(f"SubdomainOperator: A must be a CsrMatrix or an EbeMatrix, not {type(A).__name__}")
        self.A, self.comm = A, comm
        self.n = A.shape[0]
        self.device = A.device
        self.n_global = int(n_global) if n_global is not None else self.n
        self.weights = None
        if weights is not None:
            self.weights = torch.as_tensor(weights, dtype=torch.float64).to(self.device).contiguous()
        self.nbr_ranks = [int(r) for r in nbr_ranks]
        self.ovrlp = [np.asarray(v, dtype=np.int64) for v in ovrlp]
        self._halo = ctypes.c_void_p()
        self._solver = ctypes.c_void_p()
        lib = _lib.load()
        with torch.cuda.device(self.device):
            if comm is not None and comm.nranks > 1:
                # every rank builds a plan (also one without neighbours): the peer-transport import is collective
                nn = len(self.nbr_ranks)
                ranks = (ctypes.c_int32 * max(nn, 1))(*self.nbr_ranks)
                ptr = np.zeros(nn + 1, dtype=np.int64)
                ptr[1:] = np.cumsum([len(v) for v in self.ovrlp])
                idx = np.ascontiguousarray(np.concatenate(self.ovrlp)) if nn else np.zeros(1, dtype=np.int64)
                _lib.check(lib.pcgb_halo_create(comm.handle, nn, ranks, ptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                                idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), self.n,
                                                ctypes.byref(self._halo)), "pcgb_halo_create")
                if comm.transport == "peer" and comm._allgather is not None:
                    # collective: every rank exports, all-gathers and imports; if ANY rank fails (no CUDA IPC here) the whole
                    # communicator goes back to the NCCL transport so that all ranks stay on the same path
                    nb = int(lib.pcgb_halo_blob_bytes(self._halo))
                    blob = (ctypes.c_ubyte * nb)()
                    ok = lib.pcgb_halo_export(self._halo, blob) == 0
                    err = None if ok else lib.pcgb_last_error().decode()
                    blobs = comm._allgather(bytes(blob) if ok else b"")
                    if all(len(b) == nb for b in blobs):
                        buf = (ctypes.c_ubyte * (nb * comm.nranks)).from_buffer_copy(b"".join(blobs))
                        ok = lib.pcgb_halo_import(self._halo, buf) == 0
                        err = None if ok else lib.pcgb_last_error().decode()
                    else:
                        ok = False
                    if not all(o == b"1" for o in comm._allgather(b"1" if ok else b"0")):
                        comm.peer_error = err or "a peer rank could not map the halo block"
                        if comm._has_nccl:
                            comm.set_transport("nccl")
                        else:
                            raise _lib.PcgbError(f"halo exchange over peer memory is not available ({comm.peer_error}) and the communicator has no NCCL")
            create = lib.pcgb_solver_create if isinstance(A, CsrMatrix) else lib.pcgb_solver_create_ebe  # EbeMatrix: opt-in matrix-free operator
            _lib.check(create(A.handle, self._halo if self._halo else None,
                              comm.handle if comm is not None else None, ctypes.byref(self._solver)), "pcgb_solver_create")

    # -- calcMPFint on the Eff dofs (pcg_solver.py:339-342): y = A x, then the interface sum
    def apply(self, x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        y = out if out is not None else torch.empty(self.n, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().pcgb_apply(self._solver, _lib.ptr(x), _lib.ptr(y), _lib.stream_ptr()), "pcgb_apply")
        return y

    def exchange_add(self, y: torch.Tensor) -> torch.Tensor:
        """y[Ovrlp_j] += copies held by neighbour j, for all j (pcg_solver.py:303-334)."""
        if self._halo:
            with torch.cuda.device(self.device):
                _lib.check(_lib.load().pcgb_halo_exchange_add(self._halo, _lib.ptr(y), _lib.stream_ptr()), "pcgb_halo_exchange_add")
        return y

    def halo_bytes(self) -> int:
        return int(_lib.load().pcgb_halo_bytes(self._halo)) if self._halo else 0

    # -- updatePreconditioner (pcg_solver.py:346-352): 1 / (assembled diagonal)
    def jacobi(self) -> torch.Tensor:
        d = self.exchange_add(self.A.diagonal())
        out = torch.empty_like(d)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().pcgb_reciprocal(self.n, _lib.ptr(d), _lib.ptr(out), _lib.stream_ptr()), "pcgb_reciprocal")
        return out

    def solve(self, b: torch.Tensor, M: torch.Tensor | None, tol: float, maxiter: int, x0: torch.Tensor | None = None,
              w: torch.Tensor | None = None, check_every: int = 16, use_graph: bool = True, fixed_iters: bool = False,
              record_resvec: bool = False, max_stag: int = 3, time_kernels: bool = False):
        """PCG on device tensors.  Returns (x, SolveInfo); x is a new tensor (x0 is not modified)."""
        lib = _lib.load()
        dev = self.device
        assert b.is_cuda and b.dtype == torch.float64 and b.numel() == self.n
        x = x0.clone() if x0 is not None else torch.zeros(self.n, dtype=torch.float64, device=dev)
        w = w if w is not None else self.weights
        opt = _lib.Options(tol=float(tol), maxiter=int(maxiter), n_global=int(self.n_global), max_stag=int(max_stag),
                           check_every=int(check_every), use_graph=1 if use_graph else 0,
                           fixed_iters=1 if fixed_iters else 0, record_resvec=1 if record_resvec else 0,
                           time_kernels=1 if time_kernels else 0, x0_zero=1 if x0 is None else 0)
        res = _lib.Result()
        resvec = torch.zeros(maxiter + 2, dtype=torch.float64, device=dev) if record_resvec else None
        with torch.cuda.device(dev):
            _lib.check(lib.pcgb_solve(self._solver, _lib.ptr(b), _lib.ptr(M), _lib.ptr(w), _lib.ptr(x), ctypes.byref(opt),
                                      _lib.ptr(resvec), ctypes.byref(res), _lib.stream_ptr()), "pcgb_solve")
        info = SolveInfo(res.flag, res.iters, res.relres, res.normb, res.imin, res.stag, res.moresteps,
                         bool(res.too_small_tol), res.matvecs, res.launches, res.loop_ms, res.spmv_ms,
                         res.spmv_timed, res.loop_iters, res.setup_ms, res.final_ms)
        if time_kernels and res.spmv_timed > 0:
            names = ["p_update", "spmv", "halo_pack", "pq_reduce_allreduce", "halo_unpack", "fused_update", "norms_reduce_allreduce", "iteration"]
            info.phase_ms = {k: res.phase_ms[i] / res.spmv_timed for i, k in enumerate(names)}
        if record_resvec:
            info.resvec = resvec[: int(res.loop_iters) + 1].cpu().numpy()   # ||r_0|| .. ||r_k||, k = iterations executed
        return x, info

    def __del__(self):
        try:
            lib = _lib.load()
            if self._solver:
                lib.pcgb_solver_destroy(self._solver)
                self._solver = ctypes.c_void_p()
            if self._halo:
                lib.pcgb_halo_destroy(self._halo)
                self._halo = ctypes.c_void_p()
        except Exception:
            pass


def _as_operator(A, device):
    if isinstance(A, SubdomainOperator):
        return A
    if isinstance(A, CsrMatrix):
        return SubdomainOperator(A)
    if hasattr(A, "tocsr"):  # scipy sparse
        return SubdomainOperator(CsrMatrix.from_scipy(A, device=device))
    raise TypeError("solve: A must be a SubdomainOperator, CsrMatrix or scipy sparse matrix")


last_info: SolveInfo | None = None


def solve(A, b, M=None, tol: float = 1e-8, maxiter: int = 10000, x0=None, w=None, *, device="cuda",
          on_too_small_tol: str = "flag", return_info: bool = False, **kw):
    """Jacobi-PCG with the reference's (MATLAB pcg) semantics; see the module docstring.

    b / M / x0 / w may be numpy arrays (copied to the device, result returned as numpy) or CUDA tensors
    (result returned as a CUDA tensor).  on_too_small_tol="raise" reproduces the reference's
    `raise Warning('PCG : TooSmallTolerance')` (pcg_solver.py:549); the default reports MATLAB's flag 3.
    """
    global last_info
    if not torch.cuda.is_available():
        raise _lib.PcgbError("solve: no CUDA device - libpcgb200 has no CPU fallback")
    op = _as_operator(A, device)
    host_io = isinstance(b, np.ndarray)

    def dev(v):
        if v is None:
            return None
        if isinstance(v, np.ndarray):
            return torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(op.device, non_blocking=True)
        return v.to(op.device, torch.float64).contiguous()

    if isinstance(M, str):
        if M.lower() != "jacobi":
            raise ValueError("solve: M must be an inverse-diagonal vector, None or 'jacobi'")
        Md = op.jacobi()
    else:
        Md = dev(M)
    x, info = op.solve(dev(b), Md, tol, maxiter, x0=dev(x0), w=dev(w), **kw)
    last_info = info
    if info.too_small_tol and on_too_small_tol == "raise":
        raise Warning("PCG : TooSmallTolerance")
    xo = x.cpu().numpy() if host_io else x
    if return_info:
        return xo, info.flag, info.relres, info.iters, info
    return xo, info.flag, info.relres, info.iters
