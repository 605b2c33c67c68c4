#!/usr/bin/env python
"""bench.py - PCG iterations/s and SpMV GB/s (fp64) on B200, next to the CPU reference path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--block 128] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1] at N=1, the C5 stacking rule at N>1, weak scaling): every GPU owns
one box of `block`^3 trilinear hex elements (default 128^3: n = 6 390 144 free dofs, nnz = 509 597 550,
6.1 GB of CSR per GPU - far larger than the 126 MB L2) of a global mesh stacked 1x1x1 / 2x1x1 / 2x2x1 /
2x2x2, clamped at x = 0, traction on x = max; the matrix is generated on the device.  A "step" is one
PCG iteration (CSR SpMV + 2 reductions + Jacobi + AXPYs [+ halo exchange + allreduces]).

    value    subdomain-iterations/s = N * K / device time of the iteration loop (CUDA events on the solver stream, max
             over ranks): every rank advances ITS 128^3 subdomain by K PCG iterations, so the units all ranks processed
             are N*K; at N=1 this is plain PCG iterations/s, and under weak scaling v_N / (N v_1) = T_1 / T_N.
             Raw iterations/s and dof-iterations/s are reported beside it.
    parity   the first recorded residual norms ||r_k|| of a K-iteration run against the committed oracle golden of the
             same global mesh (tests/golden/hex<B>_N<N>_resvec.json <- oracle/make_golden_resvec.py); the run FAILS
             (exit code 3) when the first 10 iterations differ by more than 1e-9 relative
    e2e      the same K iterations through the public solve() with HOST buffers: b from pinned host memory,
             x back to the host, setup / verification matvecs and all host polling inside the timed region
    roofline the merge-path SpMV kernel: algorithmic bytes (12 nnz + 4|8 (n+1) + 16 n) / mean launch duration
             (event pairs around every SpMV launch of a separate K-iteration pass) against MEASURED_PEAKS.json
    cpu_baseline / --impl reference: the oracle port of the reference's numpy element-by-element PCG
             (oracle/ref_pcg.py <- pcg_solver.py:242-598) on the same mesh, one process per part like
             `mpiexec -np P`, bounded to a few iterations.
"""
from __future__ import annotations

import argparse
import json
import os

# the reference pins every BLAS to one thread per rank BEFORE numpy is imported (pcg_solver.py:10-15);
# the CPU arm forks one process per mesh part, so the same must hold here
for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
    os.environ.setdefault(_v, "1")
# stdout carries exactly one JSON line: NCCL's own banner / debug output goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "PCG iterations/sec (fp64 Jacobi-PCG, CSR SpMV) on 3-D elastostatic hex mesh, summed over the subdomains (one 128^3 subdomain per GPU)"
UNIT = "subdomain-iterations/s (= PCG iterations/s x GPUs; plain iterations/s at N=1)"
PARITY_RTOL = 1e-9      # first 10 iterations of the residual history against the oracle golden
CONCRETE_L2 = "CSR 0.88 GB in total (0.11 GB per GPU at N=8, L2-resident there): a latency-bound configuration, stated as such"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one SpMV launch of the default workload, from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json); None when no capture has been recorded."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)["spmv_dram_bytes_per_launch"]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower().startswith("active")})
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


# --------------------------------------------------------------------------------------- CPU reference arm
def _cpu_rank(rank, size, comm, ng, pgrid, iters):
    """One 'MPI rank' of the oracle port (oracle/spmd.py): its own box of the mesh as an element-by-element part,
    reductions and the interface exchange through shared memory + barriers - the reference's communication pattern
    (3 allreduces + 1 neighbour exchange per iteration, pcg_solver.py:303-334, 622-628)."""
    from oracle import ref_pcg as R
    from oracle.hex_parts import hex_box_part_spmd
    from pcg_mpi_solver_b200.hexmesh import partition_blocks
    blocks = partition_blocks(ng, pgrid)
    part = R.EbePart(hex_box_part_spmd(blocks, rank, h=1.0 / ng[0]))
    comm.setup_halo(part, comm._halo_box)
    R.update_bc([part], comm=comm)
    minv = R.Operator([part], comm).jacobi()
    nglob = 3 * (ng[0]) * (ng[1] + 1) * (ng[2] + 1)
    kw = dict(nglob=nglob, comm=comm)
    R.ref_pcg([part], minv, 1e-300, 2, **kw)                 # untimed warm-up (page faults, BLAS init)
    best = None
    for _ in range(2):                                       # two repeats, the faster one counts (host noise only ever slows it down)
        t0 = time.perf_counter()
        R.ref_pcg([part], minv, 1e-300, 1, **kw)
        t1 = time.perf_counter()
        out = R.ref_pcg([part], minv, 1e-300, 1 + iters, **kw)
        t2 = time.perf_counter()
        # difference of two runs = `iters` loop iterations only (set-up and the two residual matvecs cancel)
        dt = comm.allreduce((t2 - t1) - (t1 - t0)) / size    # the same number on every rank: all ranks pick the same repeat
        best = dt if best is None or dt < best else best
    return (best, out["Iter"], part.n)


def _cpu_rank_concrete(rank, size, comm, zp, elepart, iters):
    """One 'MPI rank' of the oracle port on a METIS part of data/concrete.zip (config C4)."""
    from oracle import ref_pcg as R
    from pcg_mpi_solver_b200.partition import partition_mesh
    sub = partition_mesh(zp, size, elepart=elepart, assemble=False)[rank]
    part = R.EbePart(sub.to_refmeshpart())
    comm.setup_halo(part, comm._halo_box)
    R.update_bc([part], comm=comm)
    minv = R.Operator([part], comm).jacobi()
    kw = dict(nglob=sub.n_global_eff, comm=comm)
    R.ref_pcg([part], minv, 1e-300, 2, **kw)
    t0 = time.perf_counter()
    R.ref_pcg([part], minv, 1e-300, 1, **kw)
    t1 = time.perf_counter()
    out = R.ref_pcg([part], minv, 1e-300, 1 + iters, **kw)
    t2 = time.perf_counter()
    return ((t2 - t1) - (t1 - t0), out["Iter"], part.n)


def _host_procs(max_procs=None):
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    p = 1
    while p * 2 <= min(cores, max_procs or 64):
        p *= 2
    return p


def cpu_reference(ng, iters, max_procs=None, units=1):
    """The oracle port on this host: the mesh is cut into P boxes (P = cores, power of two, <= 64), one process per part
    and one BLAS thread per process exactly like the reference's `mpiexec -np P` with OMP_NUM_THREADS=1
    (pcg_solver.py:10-15); the parts are coupled like the reference's ranks (shared-memory allreduce and interface
    exchange, oracle/spmd.py).  value = units * iterations/s (units = the GPU count whose global mesh this is, so that the
    CPU arm is quoted in the same subdomain-iterations/s as the GPU arm)."""
    from oracle.spmd import run_spmd
    from pcg_mpi_solver_b200.hexmesh import block_grid
    p = _host_procs(max_procs)
    while p > 1 and any(g > n for g, n in zip(block_grid(p), ng)):
        p //= 2
    res = run_spmd(p, _cpu_rank, (ng, block_grid(p), iters))
    dt = max(r[0] for r in res)
    return {"value": units * iters / dt, "unit": UNIT, "cores": p, "kind": "port", "iterations_per_s": iters / dt,
            "sample": f"{iters} PCG loop iterations (difference of a {iters}+1 and a 1 iteration run, best of 2 repeats) of the numpy element-by-element reference path "
                      f"(oracle/ref_pcg.py <- pcg_solver.py:242-598) on the same {ng[0]}x{ng[1]}x{ng[2]} hex mesh cut into {p} boxes, 1 process/box, "
                      f"1 BLAS thread each, shared-memory allreduce + interface exchange every iteration",
            "seconds": dt}


def cpu_reference_concrete(zp, iters, max_procs=8):
    """Config C4 on the host cores: data/concrete.zip cut by METIS into P parts (P <= 8 like the reference's published
    8-core run, examples/run_basic_script.bash:52), one process per part."""
    from oracle.spmd import run_spmd
    from pcg_mpi_solver_b200.metis import run_metis
    from pcg_mpi_solver_b200.model import load_mdf
    p = _host_procs(max_procs)
    ep = None
    if p > 1:
        gold = os.path.join(ROOT, "tests", "golden", f"concrete_elepart_{p}.npy")
        if os.path.exists(gold):
            ep = np.load(gold).astype(np.int64)
        else:
            m = load_mdf(zp)
            ep = run_metis(m.node_flat, m.node_offset, p)
    res = run_spmd(p, _cpu_rank_concrete, (zp, ep, iters))
    dt = max(r[0] for r in res)
    return {"value": iters / dt, "unit": UNIT, "cores": p, "kind": "port", "iterations_per_s": iters / dt,
            "sample": f"{iters} PCG loop iterations of the numpy element-by-element reference path (oracle/ref_pcg.py <- pcg_solver.py:242-598) "
                      f"on data/concrete.zip cut by METIS into {p} parts, 1 process/part, 1 BLAS thread each", "seconds": dt}


# --------------------------------------------------------------------------------------- parity helpers
def golden_resvec(block, n_gpus):
    path = os.path.join(ROOT, "tests", "golden", f"hex{block}_N{n_gpus}_resvec.json")
    if not os.path.exists(path):
        return None, path
    with open(path) as f:
        return json.load(f), path


def resvec_parity(resvec, normb, gold, path):
    """Residual history of this run against the oracle's golden of the same global mesh."""
    if gold is None:
        return {"golden": None, "checked_iterations": 0, "max_rel_err": None, "ok": None,
                "note": f"no committed golden for this mesh ({os.path.basename(path)}; oracle/make_golden_resvec.py generates it)"}
    ref = np.asarray(gold["resvec"], dtype=float)
    m = min(len(ref), len(resvec))
    rel = np.abs(np.asarray(resvec[:m]) - ref[:m]) / ref[:m]
    head = min(m, 11)                                    # ||r_0|| .. ||r_10||
    return {"golden": os.path.relpath(path, ROOT), "oracle": gold.get("oracle"), "checked_iterations": int(head - 1),
            "max_rel_err": float(rel[:head].max()), "max_rel_err_all": float(rel.max()), "compared_all": int(m - 1),
            "normb_rel_err": float(abs(normb - gold["normb"]) / gold["normb"]), "rtol": PARITY_RTOL,
            "ok": bool(rel[:head].max() <= PARITY_RTOL and abs(normb - gold["normb"]) <= PARITY_RTOL * gold["normb"])}


def preflight_parity(comm, dev, rank, world, block=6):
    """N > 1 only: the multi-GPU parity check of tests/test_gpu_multi.py inside the bench run - a 6^3-per-rank hex mesh
    (uneven cut along y) solved to 1e-12 through the same halo / all-reduce path and compared on rank 0 with the oracle's
    multi-part emulation of the reference (oracle/ref_pcg.py; used here as the checker, never timed)."""
    import torch
    import torch.distributed as dist
    from pcg_mpi_solver_b200.hexmesh import block_grid, generate_matrix, interface_lists, load_vector, partition_blocks
    from pcg_mpi_solver_b200.solver import SubdomainOperator
    pgrid = block_grid(world)
    ng = tuple(block * pgrid[a] + (1 if a == 1 else 0) for a in range(3))
    blocks = partition_blocks(ng, pgrid)
    for b_ in blocks:
        b_.h = 1.0 / ng[0]
    blk = blocks[rank]
    A = generate_matrix(blk, device=dev)
    nbr, lists, w = interface_lists(blocks, rank)
    n_global = 3 * ng[0] * (ng[1] + 1) * (ng[2] + 1)
    op = SubdomainOperator(A, comm, nbr, lists, w, n_global=n_global)
    b = load_vector(blk, device=dev)
    x, info = op.solve(b, op.jacobi(), 1e-12, 5000, check_every=8)
    gz, gy, gx = np.meshgrid(*[np.arange(blk.e0[a], blk.e0[a] + blk.ne[a] + 1) for a in (2, 1, 0)], indexing="ij")
    keep = gx.ravel() >= 1
    gnode = ((gz * (ng[1] + 1) + gy) * (ng[0] + 1) + gx).ravel()[keep]
    gdof = (3 * gnode[:, None] + np.arange(3)[None, :]).ravel()
    v = np.sin(0.37 * gdof) + 0.01 * (gdof % 7)
    y = op.apply(torch.from_numpy(v).to(dev)).cpu().numpy()
    gathered = [None] * world
    dist.gather_object({"gdof": gdof, "x": x.cpu().numpy(), "y": y}, gathered if rank == 0 else None, dst=0)
    res = None
    if rank == 0:
        from oracle import ref_pcg as R
        parts = []
        for r, bl in enumerate(blocks):
            nb, ls, ww = interface_lists(blocks, r)
            parts.append(R.CsrPart(R.hex_box_csr(bl.ng, bl.e0, bl.ne, h=bl.h), load_vector(bl, device="cpu").numpy(), nb, ls, ww, part_id=r))
        opr = R.Operator(parts)
        ref = R.ref_pcg(parts, opr.jacobi(), 1e-12, 5000, nglob=n_global)
        yrefs = opr.apply([np.sin(0.37 * g["gdof"]) + 0.01 * (g["gdof"] % 7) for g in gathered])
        ntot = 3 * (ng[0] + 1) * (ng[1] + 1) * (ng[2] + 1)
        U, Uref, Y, Yref = (np.zeros(ntot) for _ in range(4))
        for r, g in enumerate(gathered):
            U[g["gdof"]] = g["x"]; Uref[g["gdof"]] = ref["X"][r]; Y[g["gdof"]] = g["y"]; Yref[g["gdof"]] = yrefs[r]
        res = {"mesh": f"{block}^3 per rank, global {ng[0]}x{ng[1]}x{ng[2]}", "flag": info.flag, "iters": info.iters, "ref_iters": ref["Iter"],
               "x_rel_err": float(np.linalg.norm(U - Uref) / np.linalg.norm(Uref)), "y_rel_err": float(np.linalg.norm(Y - Yref) / np.linalg.norm(Yref))}
        res["ok"] = bool(info.flag == 0 and ref["Flag"] == 0 and abs(info.iters - ref["Iter"]) <= 2 and res["x_rel_err"] <= 1e-9 and res["y_rel_err"] <= 1e-13)
    del op, A
    return res


# --------------------------------------------------------------------------------------- outputs
DUMP_BUDGET_BYTES = 64_000_000


def dump_outputs(path, x, info, rank, world):
    """Writes the timed solve's outputs: x (float64, this rank's subdomain) as x.npy, or x_rank<r>.npy when N > 1, and
    solve_info.npy = [flag, iterations, relres] (float64, the same on every rank).  The files of all ranks stay within
    DUMP_BUDGET_BYTES: a rank whose x does not fit its share writes a fixed sample of it instead (seed 0, ascending dof
    indices, the same for every run of the same mesh) and those indices as <name>_index.npy."""
    os.makedirs(path, exist_ok=True)
    name = "x" if world == 1 else f"x_rank{rank}"
    xh = x.detach().cpu().numpy().astype(np.float64, copy=False)
    keep = (DUMP_BUDGET_BYTES - 4096) // world // 8
    if xh.size > keep:
        idx = np.sort(np.random.default_rng(0).choice(xh.size, keep // 2, replace=False))   # half for values, half for indices
        xh = xh[idx]
        np.save(os.path.join(path, f"{name}_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, f"{name}.npy"), xh)
    if rank == 0:
        np.save(os.path.join(path, "solve_info.npy"), np.array([info.flag, info.iters, info.relres], dtype=np.float64))


# --------------------------------------------------------------------------------------- main
def main():
    import faulthandler
    faulthandler.enable()
    faulthandler.dump_traceback_later(int(os.environ.get("PCGB_BENCH_WATCHDOG", "240")), exit=False)  # stacks on stderr if a phase hangs
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--block", type=int, default=int(os.environ.get("PCGB_BENCH_BLOCK", "128")), help="hex elements per axis per GPU")
    ap.add_argument("--cpu-iters", type=int, default=10)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workload", default="hex", choices=["hex", "hex_metis", "concrete"],
                    help="hex = block-partitioned device-generated mesh (default, C2/C5); hex_metis = same global mesh through "
                         "partition_mesh()/METIS (C3); concrete = data/concrete.zip through partition_mesh()/METIS (C4)")
    ap.add_argument("--operator", default="csr", choices=["csr", "ebe"],
                    help="csr = assembled merge-path SpMV (the north-star path, default); ebe = opt-in matrix-free operator (f1)")
    ap.add_argument("--e2e-repeats", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed solve returned (its solution x and flag / iterations / "
                         "relative residual) to DIR as .npy files, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 3)
    CE = 50 if world == 1 else 25   # iterations per CUDA graph / host poll

    from pcg_mpi_solver_b200.hexmesh import block_grid
    # the CPU arm works on the SAME global mesh as the N-GPU arm even when it is started without torchrun
    mesh_world = max(world, args.gpus if args.impl == "reference" else 1, 1)
    pgrid = block_grid(mesh_world)
    ng = tuple(args.block * pgrid[a] for a in range(3))
    config = {"workload": f"hex{args.block}^3 elements per GPU, global {ng[0]}x{ng[1]}x{ng[2]} trilinear hex elastostatics "
                          f"(E=1, nu=0.3, h=1/{ng[0]}), clamped x=0, traction on x=max, Jacobi-PCG, fixed number of iterations",
              "per_gpu_block": args.block, "process_grid": list(pgrid), "parallelism": f"dd{mesh_world}",
              "l2_policy": "inputs larger than L2 (CSR 6.1 GB per GPU vs 126 MB L2), no flush needed"}
    concrete_zip = os.path.join(ROOT, "oracle", "_ref", "concrete.zip")

    if args.impl == "reference":
        if rank != 0:
            return
        iters = max(3, min(args.steps, args.cpu_iters))
        if args.workload == "concrete":
            base = cpu_reference_concrete(concrete_zip, iters)
            config = {"workload": "data/concrete.zip (124 693 octree SBFEM elements, 616 413 free dofs), METIS-partitioned, Jacobi-PCG, fixed number of iterations",
                      "l2_policy": CONCRETE_L2}
        else:
            base = cpu_reference(ng, iters, units=mesh_world)
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": iters,
                "warmup": 0, "ms_per_step": 1e3 / base["iterations_per_s"], "higher_is_better": True, "scaling": "weak" if args.workload == "hex" else "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic" if args.workload != "concrete" else "data/concrete.zip (the reference's own model)", "config": config, "cpu_baseline": base, "iterations_per_s": base["iterations_per_s"],
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    t_start = time.time()

    def log(msg):
        if rank == 0:
            print(f"[bench +{time.time() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)

    import torch
    import torch.distributed as dist
    from pcg_mpi_solver_b200.hexmesh import generate_matrix, interface_lists, load_vector, partition_blocks
    from pcg_mpi_solver_b200.solver import Communicator, SubdomainOperator

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the b200 arm has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        comm = Communicator.from_torch_distributed(dev)

    log(f"process group / communicator up (world {world}, transport {comm.transport if comm else 'none'})")

    # ---- N > 1: small-mesh parity of the halo / all-reduce path against the oracle, before anything is timed
    preflight = preflight_parity(comm, dev, rank, world) if world > 1 else None
    if preflight is not None:
        log(f"preflight parity: {preflight}")

    if args.workload == "hex":
        setup_extra = None
        blocks = partition_blocks(ng, pgrid)
        blk = blocks[rank]
        blk.h = 1.0 / ng[0]
        for b_ in blocks:
            b_.h = blk.h
        if args.operator == "ebe":
            from pcg_mpi_solver_b200.hexmesh import generate_ebe
            A = generate_ebe(blk, device=dev)
        else:
            A = generate_matrix(blk, device=dev)
        nbr, lists, w = interface_lists(blocks, rank) if world > 1 else ([], [], None)
        n_global = 3 * ng[0] * (ng[1] + 1) * (ng[2] + 1)
        op = SubdomainOperator(A, comm, nbr, lists, w, n_global=n_global)
        b = load_vector(blk, device=dev)
    else:
        # the general pipeline: model -> METIS (run_metis.py) -> subdomain builder (partition_mesh.py) -> device assembly
        from pcg_mpi_solver_b200.partition import partition_mesh
        if args.workload == "concrete":
            zp = concrete_zip
            if not os.path.exists(zp):
                raise SystemExit("bench.py: oracle/_ref/concrete.zip is not staged (run __graft_entry__.build() in the build container)")
            ep = None
            gold = os.path.join(ROOT, "tests", "golden", f"concrete_elepart_{world}.npy")
            if os.path.exists(gold):
                ep = np.load(gold).astype(np.int64)       # the partition the reference's 8-rank golden run used
            subs = partition_mesh(zp, world, elepart=ep, assemble=False)
            config = {"workload": "data/concrete.zip (124 693 octree SBFEM elements, 616 413 free dofs), METIS-partitioned, Jacobi-PCG, fixed number of iterations",
                      "l2_policy": CONCRETE_L2}
        else:
            from pcg_mpi_solver_b200.hexmesh import hex_mdf_model
            subs = partition_mesh(hex_mdf_model(ng), world, assemble=False)
            config["workload"] = config["workload"].replace("trilinear hex elastostatics", f"trilinear hex elastostatics, METIS {world}-way element partition")
        sub = subs[rank]
        n_global = sub.n_global_eff
        torch.cuda.synchronize()
        t_asm = time.perf_counter()
        op = sub.to_operator(comm, device=dev, kind=args.operator)      # device assembly of K_i[Eff,Eff] (csrc/assemble.cuh) + SpMV plan + halo plan
        torch.cuda.synchronize()
        setup_extra = {"assemble_and_plan_s": time.perf_counter() - t_asm, "elements": int(sum(g.ck.size for g in sub.groups)), "pattern_groups": len(sub.groups)}
        A = op.A
        b = torch.from_numpy(sub.b).to(dev)
        del subs
    minv = op.jacobi()
    n = A.shape[0]
    is_csr = args.operator == "csr"
    col_released = bool(is_csr and A.release_col())      # the selected SpMV kernel does not read the 4-byte column array
    torch.cuda.empty_cache()
    log(f"operator ready ({args.operator}): n={n} halo={op.halo_bytes()} B col_released={col_released} plan={A.plan_info() if is_csr else None}")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up (also builds the CUDA graph of the iteration batch)
    op.solve(b, minv, 0.0, W, fixed_iters=True, check_every=min(W, CE))
    op.solve(b, minv, 0.0, K, fixed_iters=True, check_every=CE)
    barrier()
    log("warm-up done")

    # ---- timed region: exactly K iterations, device-timed loop
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    x, info = op.solve(b, minv, 0.0, K, fixed_iters=True, check_every=CE)
    barrier()
    loop_ms = max_over_ranks(info.loop_ms)
    log(f"timed loop: {loop_ms / K:.4f} ms/iter")
    assert info.loop_iters == K, (info.loop_iters, K)

    # ---- e2e: public API, host buffers (pinned b in, x out), everything inside the timed region; median of R repeats
    # pinned host buffers exist before the timed region (a real caller reuses them across time steps)
    b_pin = b.cpu().pin_memory()
    x_host = torch.empty(n, dtype=torch.float64).pin_memory()
    e2e_all, parts_all = [], []
    for rep in range(max(1, args.e2e_repeats)):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        barrier()
        ev[0].record()
        b_dev = b_pin.to(dev, non_blocking=True)                                                   # H2D: this solve's right-hand side
        ev[1].record()
        x_e2e, info_e = op.solve(b_dev, minv, 0.0, K, fixed_iters=True, check_every=CE)            # public operator API
        ev[2].record()
        x_host.copy_(x_e2e, non_blocking=True)                                                     # D2H: the solution
        ev[3].record()
        torch.cuda.synchronize()
        e2e_all.append(max_over_ranks(ev[0].elapsed_time(ev[3])))
        parts_all.append({"h2d_ms": ev[0].elapsed_time(ev[1]), "solve_ms": ev[1].elapsed_time(ev[2]), "d2h_ms": ev[2].elapsed_time(ev[3]),
                          "setup_ms": info_e.setup_ms, "loop_ms": info_e.loop_ms, "final_ms": info_e.final_ms})
    order = np.argsort(e2e_all)
    e2e_ms = float(e2e_all[order[len(order) // 2]])
    e2e_parts = parts_all[order[len(order) // 2]]
    clocks = sampler.stop() if rank == 0 else None
    log(f"e2e: median {e2e_ms:.1f} ms of {['%.1f' % v for v in e2e_all]}  breakdown {e2e_parts}")
    barrier()

    # ---- parity of the timed work: residual history of the same K iterations against the oracle golden
    kp = min(K, 40)
    _, info_p = op.solve(b, minv, 0.0, kp, fixed_iters=True, check_every=min(kp, CE), record_resvec=True)
    gold, gpath = golden_resvec(args.block, world) if args.workload == "hex" else (None, "n/a")
    parity = resvec_parity(info_p.resvec, info_p.normb, gold, gpath)
    parity["preflight"] = preflight
    barrier()
    log(f"parity: {parity}")

    # ---- roofline pass: same K iterations with an event pair around every SpMV launch
    _, info_k = op.solve(b, minv, 0.0, K, fixed_iters=True, check_every=CE, time_kernels=True)
    spmv_ms = info_k.spmv_ms / max(info_k.spmv_timed, 1)
    spmv_ms = max_over_ranks(spmv_ms)
    spmv_share = info_k.spmv_ms / info_k.loop_ms if info_k.loop_ms > 0 else None
    peak, peak_src = measured_peaks()
    bytes_spmv = A.spmv_bytes()
    achieved = bytes_spmv / (spmv_ms * 1e-3) / 1e9
    iter_bytes = bytes_spmv + 96 * n
    barrier()
    log(f"roofline pass: spmv {spmv_ms:.4f} ms")

    full_solve = None
    if args.workload == "concrete":   # config C4: full solve to tol 1e-8 (the reference's own run: 1085 iterations at 1e-7, 12.6 s on 8 cores)
        t0 = time.perf_counter()
        xs, fi = op.solve(b, minv, 1e-8, 10000, check_every=16)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        full_solve = {"tol": 1e-8, "flag": fi.flag, "iterations": fi.iters, "relres": fi.relres, "loop_ms": max_over_ranks(fi.loop_ms),
                      "iterations_per_s": fi.iters / (max_over_ranks(fi.loop_ms) * 1e-3), "time_to_solution_s": max_over_ranks(wall),
                      "reference_published_s": 12.6, "reference_published_note": "notebooks/solver_demo.ipynb:380-408: tol 1e-7, 1085 iterations, 8 cores"}
        barrier()

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x, info, rank, world)
        barrier()

    rc = 0
    if rank == 0:
        its = K / (loop_ms * 1e-3)
        weak = args.workload == "hex"          # hex: one more 128^3 subdomain per GPU; METIS workloads: fixed global model (strong)
        value = world * its if weak else its
        stream_bytes = A.stream_bytes() if is_csr else bytes_spmv
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": loop_ms / K,
                "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic" if args.workload != "concrete" else "data/concrete.zip (the reference's own model)",
                "config": config,      # identical keys and values in the reference arm (same workload)
                "details": dict(operator=args.operator, n_per_gpu=n, nnz_per_gpu=A.nnz if is_csr else A.nnz_equivalent, n_global=n_global,
                                plan=A.plan_info() if is_csr else {"kernel": "k_ebe_t24", "pattern_groups": 1}, col_released=col_released,
                                halo_bytes_per_exchange=op.halo_bytes(), transport=comm.transport if comm else None, metis_parts=world if args.workload != "hex" else None,
                                builder=setup_extra,
                                nvlink_bytes_per_iteration_per_gpu=(2 * op.halo_bytes() + (2 * 48 * (world - 1) if comm and comm.transport == "peer" else 0)) if comm else 0),
                "iterations_per_s": its, "dof_iterations_per_s": its * n_global,
                "e2e": {"value": (world if weak else 1) * K / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 8 * n / K, "d2h_bytes_per_step": 8 * n / K,
                        "ms": e2e_ms, "repeats_ms": e2e_all, "breakdown_ms": e2e_parts, "fraction_of_value": (K / (e2e_ms * 1e-3)) / its,
                        "note": "median of the repeats; one solve() of K iterations: pinned-host b -> device, ||b|| + rho0, K iterations, the true-residual "
                                "matvec of the non-converged exit (pcg_solver.py:568-582), host polling, x -> pinned host"},
                "gpu_launches": int(info.launches),
                "clocks": clocks,
                "roofline": {"kernel": ({0: "k_spmv_merge", 1: "k_spmv_staged", 2: "k_spmv_persist"}[A.plan_info()["staged"]] + " (merge-path CSR SpMV, fp64)") if is_csr else "k_ebe_t24 (matrix-free EBE operator, fp64; bytes = its own 108 B/element, not the CSR figure)", "bound": "hbm", "achieved": achieved, "peak": peak,
                             "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic() if is_csr else None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": bytes_spmv, "streamed_bytes_per_launch": stream_bytes,
                             "streamed_GBps": stream_bytes / (spmv_ms * 1e-3) / 1e9, "streamed_frac_of_peak": stream_bytes / (spmv_ms * 1e-3) / 1e9 / peak,
                             "mean_launch_ms": spmv_ms, "launches_timed": int(info_k.spmv_timed),
                             "spmv_share_of_step": spmv_share, "phase_ms_per_iteration": info_k.phase_ms,
                             "iteration": {"algorithmic_bytes": iter_bytes, "achieved_GBps": iter_bytes / (loop_ms / K * 1e-3) / 1e9,
                                           "frac": iter_bytes / (loop_ms / K * 1e-3) / 1e9 / peak}},
                "parity": parity, "full_solve": full_solve}
        if world == 1 and not args.no_cpu and args.workload in ("hex", "concrete"):
            try:
                line["cpu_baseline"] = cpu_reference(ng, max(1, args.cpu_iters)) if args.workload == "hex" else cpu_reference_concrete(concrete_zip, max(1, args.cpu_iters))
            except Exception as e:  # the baseline is a report, never a reason to lose the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line))
        if parity.get("ok") is False or (preflight is not None and not preflight.get("ok", False)):
            print(f"bench.py: PARITY FAILURE: {parity}", file=sys.stderr)
            rc = 3
    if world > 1:
        t = torch.tensor([rc], dtype=torch.int32, device=dev)
        dist.broadcast(t, src=0)
        rc = int(t.item())
        dist.barrier()
        del op
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


if __name__ == "__main__":
    main()
