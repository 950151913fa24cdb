#!/usr/bin/env python
"""bench.py -- the adjoint hot path on B200: dRdW^T*psi throughput (GCells/s) and adjoint-solve wall time.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--cells C] [--scaling weak|strong] [--dump-outputs DIR]

A "step" is one matrix-free product y = diag(n) (dR/dW)^T psi over the whole mesh (the body of the reference's GMRES
shell-matrix callback, DASolver.C:1364-1409).  Workload: BASELINE.json configs[1], "DASimpleFoam NACA0012 SA turbulence
1M cells": a synthetic O-grid 1440x720x1 = 1 036 800 cells (the reference ships no mesh), tile-major cell numbering
(16x12 tiles, the order a bandwidth-reducing renumbering leaves), analytic boundary-layer state + 0.1 % seeded noise.
With N GPUs: weak scaling (default; N x cells, RCB partitions) or strong scaling (--scaling strong; the same mesh).
The adjoint solve (preconditioner assembly + Krylov solve of [dRdW]^T psi = dFdW) runs at every N.
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NORM_STATES = dict(U=10.0, p=50.0, nuTilda=1e-3, phi=1.0)
TILE = (16, 12)  # cells per tile of the generator's tile-major numbering (ni % 16 == 0, nj % 12 == 0)


TILE3 = (8, 6, 4)  # bricks of the 3-D wing mesh (BASELINE config 4)


def grid_for(cells):
    """O-grid ni x nj = 2 nj x nj closest to `cells` with nj a multiple of 24 (whole 16x12 tiles)."""
    nj = max(24, int(round((cells / 2.0) ** 0.5 / 24.0)) * 24)
    return 2 * nj, nj


def grid3_for(cells):
    """Swept tapered wing (BASELINE config 4): ni x nj x nk = 2 nj x nj x nk hexahedra, nk ~ 1.1 nj, whole 8x6x4 bricks."""
    nj = max(12, int(round((cells / 2.2) ** (1.0 / 3.0) / 12.0)) * 12)
    nk = max(4, int(round(cells / (2.0 * nj * nj) / 4.0)) * 4)
    return 2 * nj, nj, nk


class ClockSampler:
    def __init__(self):
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def start(self):
        def run():
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            while not self._stop.is_set():
                try:
                    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i", "0"],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
                except Exception:
                    pass
                self._stop.wait(0.1)
        self._t = threading.Thread(target=run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arms.  "port": the oracle restatement of the reference's algorithm (tape recorded once, evaluated per product =
# CoDiPack's tape.evaluate()).  "handcoded": the engine's own hand-derived reverse sweep compiled for the host
# (tests/hostsim) -- the strong CPU baseline.  One process per usable core, each on a partition-sized O-grid of the same
# physics: cells_total / P cells per process, as an MPI run of the reference on the bench mesh would have.
# ---------------------------------------------------------------------------------------------------
_WORKER = r"""
import sys, time, json
sys.path.insert(0, %(root)r)
import numpy as np
from dafoam_b200 import cases
ni, nj, engine = %(ni)d, %(nj)d, %(engine)r
m = cases.naca0012_ogrid(ni=ni, nj=nj, nk=1)
if engine == "port":
    from oracle.pyoracle import Oracle, synthetic_state
    o = Oracle(m, cases.default_bcs_naca(), normalizeStates=%(ns)r)
    W = synthetic_state(m, o.geometry("C"), o.geometry("Sf"))
    t0 = time.time(); o.record(W); trec = time.time() - t0
    psi = np.random.default_rng(4321).uniform(-1, 1, o.ndof)
    def product(): o.jtvec(psi)
else:
    import tempfile
    from dafoam_b200.pyDASolvers import pyDASolvers
    from oracle.pyoracle import synthetic_state
    d = tempfile.mkdtemp(prefix="dab_cpu_")
    cases.write_case(d, m, cases.default_bcs_naca(), binary=True)
    sol = pyDASolvers("DASimpleFoam -python", dict(normalizeStates=%(ns)r), caseDir=d, _lib_path=%(hostsim)r)
    n = sol.getNLocalAdjointStates()
    yv = np.zeros(m.n_cells); sol.getOFField("yWall", "scalar", yv)
    W = cases.boundary_layer_state(m, yv, noise=0.001)
    t0 = time.time(); sol.updateOFFields(W); R = np.zeros(n); sol.getResiduals(R); trec = time.time() - t0
    psi = np.random.default_rng(4321).uniform(-1, 1, n); y = np.zeros(n)
    def product(): sol.calcdRdWTPsiAD(psi, y)
product()
print("READY %%d %%.4f" %% (m.n_cells, trec), flush=True)
for line in sys.stdin:
    reps = int(line.split()[1])
    t0 = time.time()
    for _ in range(reps):
        product()
    print(json.dumps(dict(seconds=time.time() - t0, reps=reps)), flush=True)
"""


def usable_cores():
    """Cores this process may really use: CPU affinity, the cgroup quota, and physical (not hyper-threaded) cores."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    src = "affinity %d" % n
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            quota = max(1, int(float(q[0]) / float(q[1])))
            if quota < n:
                n, src = quota, src + ", cgroup quota %d" % quota
    except Exception:
        pass
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys and phys < n:
            n, src = phys, src + ", physical cores %d" % phys
    except Exception:
        pass
    return max(1, n), src


class CpuArm:
    """P persistent worker processes; every run() is one bounded sample: `reps` products on each partition."""

    def __init__(self, cells_total, engine="port", procs=None):
        self.cores, self.cores_src = usable_cores()
        self.P = procs or self.cores
        self.engine = engine
        nj = max(8, int(round((cells_total / self.P / 2.0) ** 0.5 / 2.0)) * 2)
        self.ni, self.nj = 2 * nj, nj
        code = _WORKER % dict(root=ROOT, ni=self.ni, nj=self.nj, engine=engine, ns=NORM_STATES,
                              hostsim=os.path.join(ROOT, "tests", "hostsim", "libdab200_hostsim.so"))
        self.procs = [subprocess.Popen([sys.executable, "-c", code], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
                      for _ in range(self.P)]
        self.cells, self.trec = 0, 0.0
        for p in self.procs:
            tok = p.stdout.readline().split()
            assert tok and tok[0] == "READY", "CPU worker failed to start"
            self.cells += int(tok[1])
            self.trec = max(self.trec, float(tok[2]))
        self.solo = None

    def _go(self, procs, reps):
        t0 = time.time()
        for p in procs:
            p.stdin.write("go %d\n" % reps)
            p.stdin.flush()
        res = [json.loads(p.stdout.readline()) for p in procs]
        return time.time() - t0, res

    def run(self, reps):
        if self.solo is None:  # one process alone: the undisturbed per-product time
            _, r = self._go(self.procs[:1], max(2, reps // 2))
            self.solo = r[0]["seconds"] / r[0]["reps"]
        wall, res = self._go(self.procs, reps)
        per = max(r["seconds"] for r in res) / reps
        slow = per / self.solo if self.solo > 0 else None
        if slow and slow > 3.0:
            sys.stderr.write("[bench] WARNING: CPU arm: a product takes %.1fx longer with %d processes running than alone "
                             "(memory-bound tape / oversubscribed cores)\n" % (slow, self.P))
        kind = "port" if self.engine == "port" else "port-handcoded"
        what = ("oracle port of the reference's CoDiPack tape-evaluate matvec" if self.engine == "port"
                else "the engine's hand-derived reverse sweep compiled for the host (tests/hostsim)")
        return dict(value=self.cells * reps / wall / 1e9, unit="GCells/s", cores=self.P, kind=kind, cores_source=self.cores_src,
                    sample="%d processes x %d-cell O-grid partition (%dx%d) x %d products (%s; wall %.2f s)"
                           % (self.P, self.cells // self.P, self.ni, self.nj, reps, what, wall),
                    cells_total=self.cells, seconds_per_product=wall / reps, seconds_per_product_one_process_alone=self.solo,
                    slowdown_all_vs_alone=slow, oversubscribed=bool(slow and slow > 3.0), record_seconds=self.trec)

    def close(self):
        for p in self.procs:
            try:
                p.stdin.close()
            except Exception:
                pass
        for p in self.procs:
            p.wait()


def run_reference(args, rank):
    """--impl reference: the reference's algorithm for this path on the host cores (oracle port; the reference itself needs
    OpenFOAM + CoDiPack + PETSc, DESIGN.md section 9).  Rank 0 only; the other ranks exit without work."""
    if rank != 0:
        return
    ni, nj = grid_for(args.cells)
    arm = CpuArm(ni * nj, "port")
    if args.warmup > 0:
        arm.run(args.warmup)
    last = arm.run(args.steps)  # one step = one product on every partition at once
    arm.close()
    v = last["value"]
    out = {"impl": "reference", "metric": "dRdWTPsi_GCells_per_s", "value": v, "unit": "GCells/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * last["seconds_per_product"], "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "%s NACA0012 SA %dx%dx1 O-grid, %d cells as %d partitions of %d cells on %d host cores"
                                  % (args.solver, ni, nj, ni * nj, last["cores"], last["cells_total"] // last["cores"], last["cores"])},
           "cpu_baseline": last,
           "e2e": {"value": v, "unit": "GCells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


# ---------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(obj):
    """The one JSON line goes to the real stdout; everything else any library prints (e.g. NCCL's version banner)
    was redirected to stderr at start-up."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


DUMP_BYTES = 60 << 20  # all arrays of --dump-outputs together: under 64 MB with the .npy headers


def dump_outputs(d, arrays):
    """Write every array as d/<name>.npy in float64, the arrays sharing DUMP_BYTES equally.  A longer array is stored as its
    entries at np.sort(np.random.default_rng(0).choice(size, share, replace=False)): the same indices on every run of the same
    arguments, so that two builds can be compared entry for entry."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_BYTES // (8 * max(1, len(arrays)))
    info = {}
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        size = a.size
        if size > share:
            a = a[np.sort(np.random.default_rng(0).choice(size, share, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)
        info[name] = {"size": size, "stored": int(a.size), "sampled": size > share}
    return {"dir": os.path.abspath(d), "arrays": info}


def global_state(mesh, comp, U0c, thermo):
    """Smooth analytic boundary-layer state (+0.1 % seeded noise) on the global mesh -- SURVEY.md section 8d."""
    from scipy.spatial import cKDTree
    from dafoam_b200 import cases
    Sf, Cf = cases.quad_face_geometry(mesh)
    wall = [p for p in mesh.patches if p["type"] == "wall"][0]
    nIF = mesh.n_internal_faces
    # cell centres as the mean of the face centres (bincount: np.add.at is ~50x slower at 10^7 faces)
    nC = mesh.n_cells
    cnt = np.bincount(mesh.owner, minlength=nC) + np.bincount(mesh.neighbour, minlength=nC)
    Cc = np.stack([np.bincount(mesh.owner, weights=Cf[:, k], minlength=nC) + np.bincount(mesh.neighbour, weights=Cf[:nIF, k], minlength=nC)
                   for k in range(3)], axis=1) / cnt[:, None]
    yw = cKDTree(Cf[wall["start"]:wall["start"] + wall["size"]]).query(Cc, workers=-1)[0]
    Wg = cases.boundary_layer_state(mesh, yw, U0=U0c if comp else (10.0, 0.0, 0.0), seed=1234, noise=0.001)
    if comp:
        Wg = cases.to_compressible_state(mesh, Wg, thermo)
    return Wg


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--cells", type=int, default=1036800)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = N x cells (fixed work per GPU, default), strong = the same mesh on every N")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-solve", action="store_true")
    ap.add_argument("--no-gmres", action="store_true", help="skip the GMRES leg of the adjoint solve (the reference's KSP)")
    ap.add_argument("--gmres-multi", action="store_true", help="run the GMRES leg on several GPUs too")
    ap.add_argument("--restart", type=int, default=1500)
    ap.add_argument("--pc-level", type=int, default=None, help="pcConLevel of dRdWTPC (default 3 on the 2-D O-grid, 2 on the 3-D wing: a level-3 ball holds 63 hexahedra)")
    ap.add_argument("--pc-block", type=int, default=0,
                    help="adjEqnOption.pcBlockCells: block-Jacobi ILU(0) with natural order inside blocks of that many cells (0: multicolour)")
    ap.add_argument("--coarse", type=int, default=2000)
    ap.add_argument("--pc-storage", default="fp32", choices=["fp32", "fp64"],
                    help="adjEqnOption.pcStorage: fp32 copy of the ILU factors for the triangular solves (operator and vectors stay fp64)")
    ap.add_argument("--idr-s", type=int, default=8)
    ap.add_argument("--max-iters", type=int, default=3000)
    ap.add_argument("--mesh", default="ogrid2d", choices=["ogrid2d", "wing3d", "passage"],
                    help="wing3d: BASELINE config 4, a swept tapered NACA0012 wing between two symmetry planes, fully 3-D hexahedra (use --cells 5000000 --gpus 4); "
                         "passage: BASELINE config 5's shape, one passage of an annular rotor row with cyclic sides and an MRF zone (use --solver DATurboFoam)")
    ap.add_argument("--solver", default="DASimpleFoam", choices=["DASimpleFoam", "DARhoSimpleFoam", "DATurboFoam"],
                    help="DARhoSimpleFoam: BASELINE config 3 (compressible airfoil; use --cells 2000000); DATurboFoam: config 5 (with --mesh passage)")
    ap.add_argument("--reference-schemes", action="store_true",
                    help="the schemes the reference's NACA0012 cases select: div(phi,U) linearUpwindV and nutUSpaldingWallFunction on the wing "
                         "(the RevB<6,7> / FwdB<6,7> kernel variants instead of the light <6,0> ones); not the default workload")
    ap.add_argument("--primal-iters", type=int, default=None,
                    help="run that many SIMPLE iterations (solvePrimal on the GPU) from the synthetic state before the adjoint legs (1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the run computed as DIR/<name>.npy (float64, rank 0's local vectors): dRdWTPsi, the y the last timed "
                         "product returned, and adjoint_psi_<leg>, the solution of each adjoint-solve leg; see dump_outputs for the size bound")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)

    from dafoam_b200 import cases
    from dafoam_b200.pyDASolvers import pyDASolvers

    ncell_target = args.cells * (world if args.scaling == "weak" else 1)
    wing = args.mesh == "wing3d"
    passage = args.mesh == "passage"
    if args.pc_level is None:
        args.pc_level = 2 if (wing or passage) else 3
    if args.primal_iters is None:
        # the synthetic passage state (a profile with slip at a hub that rotates under it) is far from any flow: ILU(0) of its Jacobian
        # is unstable (GMRES stagnates, IDR diverges at 65k cells on the host build); after 300 SIMPLE iterations it is a flow
        args.primal_iters = 300 if passage else 0
    if passage:
        # 36 passages (10 degree pitch); radial : pitchwise : axial cell counts 1 : 1 : 2
        nj = ni = max(4, int(round((ncell_target / 2.0) ** (1.0 / 3.0))))
        nk = max(4, int(round(ncell_target / float(ni * nj))))
        tile = (1, 1, 1)
    elif wing:
        ni, nj, nk = grid3_for(ncell_target)
        tile = TILE3
    else:
        (ni, nj), nk = grid_for(ncell_target), 1
        tile = TILE
    t_setup = time.time()
    comp = args.solver in ("DARhoSimpleFoam", "DATurboFoam")
    U0c = (100.0, 0.0, 0.0)  # M ~ 0.29 at 300 K
    thermo = cases.default_thermo(energy="sensibleEnthalpy" if args.solver == "DATurboFoam" else "sensibleInternalEnergy") if comp else None
    partitioned = world > 1 or passage  # the engine's state vector is then a local one (ghost / image slots), filled from a global state
    # rank 0 generates the mesh, writes the case (binary polyMesh) and, on several GPUs, the global state; the other ranks
    # only read: their own engine reads the polyMesh and keeps its partition, the state slice comes from the shared file
    mesh = None
    info = [None, None, 0, 0]
    ref_kw = dict(div_u="bounded Gauss linearUpwindV grad(U)") if args.reference_schemes else {}
    if rank == 0 and passage:
        mesh = cases.annular_passage(nr=ni, nt=nj, nz=nk, r0=0.2, r1=0.35, lz=0.3, n_sectors=36)
        case_dir = tempfile.mkdtemp(prefix="dab_bench_")
        Uax = 100.0 if comp else 10.0
        bcs = cases.default_bcs_passage(Uin=(0.0, 0.0, Uax))
        mrf = dict(cellZone="rotor", cells=np.arange(mesh.n_cells), origin=(0.0, 0.0, 0.0), axis=(0.0, 0.0, 1.0), omega=300.0 if comp else 30.0,
                   nonRotatingPatches=["inlet", "outlet", "shroud"])
        if comp:
            cases.write_case(case_dir, mesh, cases.compressible_bcs(bcs), binary=True, thermo=thermo, mrf=mrf)
        else:
            cases.write_case(case_dir, mesh, bcs, binary=True, mrf=mrf)
        n_merged = cases.merged_face_order(mesh).size
        info = [case_dir, None, mesh.n_cells, n_merged]
        if world > 1:
            from dafoam_b200.pyDASolvers import nccl_unique_id
            info[1] = nccl_unique_id()
        np.save(os.path.join(case_dir, "W_global.npy"), cases.passage_state(mesh, Uax=Uax, thermo=thermo, n_sectors=36))
    elif rank == 0:
        if wing:
            mesh = cases.naca0012_ogrid(ni=ni, nj=nj, nk=nk, span=3.0, sweep=0.5, taper=0.5, radius=15.0, tile=tile)
        else:
            mesh = cases.naca0012_ogrid(ni=ni, nj=nj, nk=1, tile=tile)
        case_dir = tempfile.mkdtemp(prefix="dab_bench_")
        if comp:
            cases.write_case(case_dir, mesh, cases.compressible_bcs(cases.default_bcs_naca(U0=U0c, wall_function=args.reference_schemes)), binary=True,
                             thermo=thermo, **ref_kw)
        else:
            cases.write_case(case_dir, mesh, cases.default_bcs_naca(wall_function=args.reference_schemes), binary=True, **ref_kw)
        info = [case_dir, None, mesh.n_cells, mesh.n_faces]
        if world > 1:
            from dafoam_b200.pyDASolvers import nccl_unique_id
            info[1] = nccl_unique_id()
            np.save(os.path.join(case_dir, "W_global.npy"), global_state(mesh, comp, U0c, thermo))
    if world > 1:
        dist.broadcast_object_list(info, src=0)
    case_dir, uid, n_cells_g, n_faces_g = info
    t_mesh = time.time() - t_setup
    fn = {"CD": {"type": "force", "source": "patchToFace", "patches": ["hub" if passage else "wing"], "directionMode": "fixedDirection",
                 "direction": [0.0, 0.0, 1.0] if passage else [1.0, 0.0, 0.0], "scale": 1.0}}
    ns_opt = dict(U=100.0, p=101325.0, T=300.0, nuTilda=1e-3, phi=1.0) if comp else NORM_STATES
    adj_opt = dict(gmresRelTol=1e-6, gmresMaxIters=args.max_iters, gmresRestart=args.restart, printInfo=1, pcConLevel=args.pc_level,
                   coarseAggregates=args.coarse, pcBlockCells=args.pc_block, pcStorage=args.pc_storage, tileCells=int(np.prod(tile)))
    opts = dict(normalizeStates=ns_opt, function=fn, primalMaxIters=max(args.primal_iters, 1), primalMinResTol=1e-8, printInterval=100,
                adjEqnOption=adj_opt)
    sol = pyDASolvers(args.solver + " -python", opts, caseDir=case_dir, device=local_rank, rank=rank, nRanks=world, ncclUniqueId=uid)
    n = sol.getNLocalAdjointStates()
    nC = sol.getNLocalCells()
    if not partitioned:
        y_ = np.zeros(nC)
        sol.getOFField("yWall", "scalar", y_)
        W = cases.boundary_layer_state(mesh, y_, U0=U0c if comp else (10.0, 0.0, 0.0), seed=1234, noise=0.001)
        if comp:
            W = cases.to_compressible_state(mesh, W, thermo)
    else:
        Wg = np.load(os.path.join(case_dir, "W_global.npy"), mmap_mode="r")
        W = np.ascontiguousarray(Wg[sol.localStateIndex(n_cells_g, n_faces_g, compressible=comp)])
        del Wg
    del mesh
    sol.updateOFFields(W)
    t_setup = time.time() - t_setup
    primal = None
    if args.primal_iters > 0 and (world == 1 or passage):
        # the step before the path (solve_nonlinear): SIMPLE iterations on the device, then the adjoint at that state
        pfail = sol.solvePrimal()
        ps = sol.primalStats
        sol.getOFFields(W)
        sol.updateOFFields(W)  # the states the adjoint legs pass to calcJacTVecProduct are then the resident ones (no second assembly)
        primal = {"iterations": ps.iterations, "seconds": ps.seconds, "max_residual": ps.max_residual, "converged": int(ps.converged),
                  "fail": pfail, "p_iterations": ps.p_iterations, "ms_per_iteration": 1e3 * ps.seconds / max(ps.iterations, 1),
                  "CD": sol.calcFunction("CD")}

    # pinned host buffers for the end-to-end (host-buffer) leg
    psi_h = torch.empty(n, dtype=torch.float64).pin_memory()
    y_h = torch.empty(n, dtype=torch.float64).pin_memory()
    psi = psi_h.numpy()
    y = y_h.numpy()
    psi[:] = np.random.default_rng(4321 + rank).uniform(-1, 1, n)
    sol.benchSetVector(psi)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg (value): K products, CUDA events on the solver's stream inside the C ABI
    sol.benchDevice(0, args.warmup)
    sampler = ClockSampler()
    if rank == 0:
        sampler.start()
    barrier()
    ms, launches = sol.benchDevice(0, args.steps)
    barrier()
    per_kernel = {name: sol.benchDevice(which, max(5, args.steps // 5))[0] for name, which in (("RevA", 2), ("RevB", 3), ("RevC", 4))}
    ms_fwd, _ = sol.benchDevice(1, max(5, args.steps // 5))

    # ---- end-to-end leg: the public call with HOST buffers (H2D psi + 3 kernels + D2H y every step)
    for _ in range(3):
        sol.calcdRdWTPsiAD(psi, y)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sol.calcdRdWTPsiAD(psi, y)
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    outputs = {"dRdWTPsi": y.copy()}

    # max over ranks
    tt = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = float(tt[0]), float(tt[1])

    # ---- adjoint solve at every N: dRdWTPC assembly + factorisation, then [dRdW]^T psi = dFdW to 1e-6.  Two Krylov legs on the
    # same preconditioner: IDR(s) (adjEqnOption.kspType idrs, an extension: short recurrences, no orthogonalisation against the whole
    # basis) and GMRES, the reference's KSP (its restart bounded by the basis that fits next to the preconditioner in HBM)
    adjoint = None
    if not args.no_solve:
        try:
            from dafoam_b200.pyDASolvers import Mat, KSP
            barrier()
            t0 = time.perf_counter()
            pc = Mat()
            sol.calcdRdWT(1, pc)
            ksp = KSP()
            sol.createMLRKSPMatrixFree(pc, ksp)
            barrier()
            t_pc = time.perf_counter() - t0
            dFdW = np.zeros(n)
            sol.calcJacTVecProduct("states", "stateVar", W, "CD", "function", np.array([1.0]), dFdW)
            adjoint = {"pc_s": t_pc, "tolerance": 1e-6}

            def leg(name, ksp_opts):
                sol.updateDAOption(dict(adjEqnOption=ksp_opts))
                x = np.zeros(n)
                barrier()
                t1 = time.perf_counter()
                fail = sol.solveLinearEqn(ksp, dFdW, x)
                barrier()
                dt = time.perf_counter() - t1
                tm = torch.tensor([dt], dtype=torch.float64, device="cuda")
                if world > 1:
                    dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                st = ksp.stats
                return x, {"method": name, "wall_s": t_pc + float(tm[0]), "solve_s": float(tm[0]), "fail": fail, "iterations": st.iterations,
                           "rel_residual": st.final_residual / st.initial_residual if st.initial_residual else None,
                           "n_matvec": st.n_matvec, "device_s": st.solve_seconds}

            psi_i, adjoint["idrs"] = leg("IDR(%d)" % args.idr_s, dict(kspType="idrs", idrS=args.idr_s, gmresMaxIters=3 * args.max_iters))
            outputs["adjoint_psi_idrs"] = psi_i
            best = adjoint["idrs"]
            if not args.no_gmres and (world == 1 or args.gmres_multi):  # the GMRES leg (25 s and a 110 GB basis at 1M cells) runs on one GPU only by default
                free_b = torch.cuda.mem_get_info()[0]
                m_fit = int(0.8 * free_b / (8.0 * n)) - 8
                restart = max(30, min(args.restart, m_fit))
                try:
                    psi_g, adjoint["gmres"] = leg("GMRES(%d), the reference's KSP" % restart,
                                                  dict(kspType="gmres", gmresRestart=restart, gmresMaxIters=args.max_iters))
                    outputs["adjoint_psi_gmres"] = psi_g
                    dn = float(np.linalg.norm(psi_g))
                    adjoint["idrs"]["psi_rel_diff_vs_gmres"] = float(np.linalg.norm(psi_i - psi_g)) / dn if dn > 0 else None
                    if adjoint["gmres"]["fail"] == 0 and (best["fail"] or adjoint["gmres"]["wall_s"] < best["wall_s"]):
                        best = adjoint["gmres"]
                except Exception as e:
                    adjoint["gmres"] = {"error": str(e)}
            # headline fields = the faster converged leg
            for k in ("method", "wall_s", "solve_s", "fail", "iterations", "rel_residual", "n_matvec"):
                adjoint[k] = best[k]
        except Exception as e:  # reported, never hidden
            adjoint = {"error": str(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    traffic, traffic_src = None, None
    tf = os.path.join(ROOT, "profiles", "r02_ncu_kernels_dram.json")
    if os.path.exists(tf) and world == 1 and not comp:
        tj = json.load(open(tf))
        if tj.get("cells") == n_cells_g:
            traffic = sum(tj[k]["dram__bytes_read.sum"] + tj[k]["dram__bytes_write.sum"] for k in ("RevA", "RevB", "RevC"))
            traffic_src = "profiles/r02_ncu_kernels_dram.json (ncu dram__bytes_read+write of RevA+RevB+RevC, same workload, commit %s)" % tj.get("commit")
    alg = sol.algorithmicBytes(0)
    achieved = alg / (ms_max * 1e-3) / 1e9
    nC_global = sol.getNGlobalCells()
    value = nC_global / (ms_max * 1e-3) / 1e9
    out = {
        "metric": "dRdWTPsi_GCells_per_s", "value": value, "unit": "GCells/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s %s SA %s %dx%dx%d (%s tiles), %d cells global, %d cells / %d DOF "
                               "on this GPU; adjoint matvec dRdW^T*psi; working set per product ~%.0f MB >> 126 MB L2 (no explicit flush)"
                               % (args.solver, "annular rotor passage (36 per row), cyclic sides + MRF zone," if passage else
                                  ("NACA0012 (linearUpwindV + Spalding wall function)" if args.reference_schemes else "NACA0012"),
                                  "radial x pitchwise x axial" if passage else ("swept tapered wing, 3-D O-grid" if wing else "O-grid, tile-major cell numbering"),
                                  ni, nj, nk, "x".join(str(t) for t in tile),
                                  nC_global, nC, n, (alg + 60 * 8 * nC) / 1e6),
                   "parallelism": ("domain decomposition (RCB) over %d GPUs, NCCL ghost-cell exchange" % world) if world > 1 else "single GPU",
                   "setup_s": t_setup, "setup_mesh_generation_s": t_mesh},
        "gpu_launches": launches,
        "e2e": {"value": nC_global / (e2e_ms_max * 1e-3) / 1e9, "unit": "GCells/s", "ms_per_step": e2e_ms_max,
                "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 8 * n,
                "call": "pyDASolvers.calcdRdWTPsiAD(psi_host, y_host) -> dab_drdwt_mat_vec (pinned host buffers)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_product": alg,
                     "kernels_ms": per_kernel, "forward_R_ms": ms_fwd,
                     "note": "one product = RevA+RevB+RevC; achieved = algorithmic bytes of the product / its device time"},
        "adjoint_solve": adjoint,
        "primal_solve": primal,
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1 and not comp and not wing and not passage:
        try:
            arm = CpuArm(nC_global, "port")
            out["cpu_baseline"] = arm.run(10)
            arm.close()
            # perfectly scaled bound: every core as fast as one process alone (the ratio to quote beside the measured one)
            cb = out["cpu_baseline"]
            cb["value_if_perfectly_scaled"] = cb["cells_total"] / cb["seconds_per_product_one_process_alone"] / 1e9
            arm = CpuArm(nC_global, "handcoded")
            out["cpu_baseline_handcoded"] = arm.run(10)
            arm.close()
            # config 1 of BASELINE.json (the reference's own ~5k-cell case on ONE CPU rank): the same port on one core
            arm = CpuArm(5832, "port", procs=1)
            out["cpu_baseline_1core"] = arm.run(10)
            arm.close()
        except Exception as e:
            out["cpu_baseline"] = {"error": str(e)}
    if args.dump_outputs:
        out["dumped_outputs"] = dump_outputs(args.dump_outputs, outputs)
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
