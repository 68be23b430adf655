#!/usr/bin/env python
"""bench.py -- headline benchmark of the barrier-Newton hot path (BASELINE.json configs[1]).

Workload: `mgb_solve(assemble(amg(subdivide(fem2d_P1(), 10)); p=1.5))`, n = 1 572 864 broken nodes
(DOF), Float64, synthetic default problem (src/mgb.jl:587-613).  One *step* = one whole solve: the
t-ramp with every Newton iteration, Hessian assembly, V-cycle PCG solve and line search on the GPU.

  value  = DOF * Newton-steps / s with the problem already resident in HBM (handle created before the timed
           region; each step restarts from the boundary data g).
  e2e    = the same metric through the public API `mgbx.solver.mgb_solve(prob)` with HOST buffers: handle
           creation (H2D of every grid / operator / hierarchy + plan build), the solve, and the D2H of z.
           The host buffers are in the reference's own layout (Julia arrays are column-major; operator blocks
           p x p x N), which is what the C ABI takes: the per-geometry conversion of the Python mirror's
           operator blocks is cached on the geometry, so only the first (untimed warm-up) call pays it.
  parity = the timed solve against the committed CPU-oracle fixture of the SAME workload
           (tests/golden/size_fem2d_P1_L<L>_p1.5.npz): relative L2 error of z, relative error of the final
           objective, Newton-step totals.  For N > 1 the same, from the partitioned solve.
  roofline     = the dominant kernel class, timed live with CUDA events on the library's stream (profile pass).
  same_config  = this GPU path at the levels the CPU arms run (L = 7 for cpu_baseline, L = 8 for `--impl reference`),
                 so that like-for-like pairs exist beside the L = 10 headline.
  cpu_baseline = the CPU oracle (NumPy/SciPy, SuperLU; 1 thread), ONE full-tolerance solve at L = 7 (about 30 s).

`--impl reference` times the CPU oracle arm alone: ONE full-tolerance solve at L = 8 (n = 98 304, about 2 minutes; the
path is deterministic, so it is run once, not warmup + steps times).  The reference itself is Julia; there is no Julia here
(baseline/run_reference.jl is the script for a box that has it).
N > 1 (torchrun): ONE solve, elements partitioned over the ranks (partition.py), max-over-ranks time ("strong").

`--dump-outputs DIR` writes what the last timed solve returned (z, z_unfinalized and the t-ramp history of SOL_main) as
float64 DIR/<name>.npy, so that two builds can be compared output for output: the problem is synthetic and deterministic,
so the same arguments give the same inputs on every run.
The bench writes nothing into the tree it runs from (which may be read-only): no bytecode, and numba's cache of the host-side
AMG setup goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

METRIC = "mgb_solve DOF*Newton-steps/s (fem2d_P1 ~1.6M DOF, p=1.5)"
UNIT = "DOF*Newton-steps/s"
REF_L = 8          # --impl reference: largest level whose single full-ramp oracle solve takes ~2 minutes
CPU_L = 7          # cpu_baseline leg of the default run (~30 s)
DUMP_BYTES = 64 << 20


def build_problem(L, p):
    import mgbx  # noqa: F401
    from mgbx import geometry as G, hierarchy as H, problem as P
    return P.assemble(H.amg(G.subdivide(G.fem2d_P1(), L)), p=p)


def workload_name(L, p, n=None):
    return "mgb_solve(assemble(amg(subdivide(fem2d_P1(),%d)); p=%g))%s" % (L, p, "" if n is None else ": n=%d broken nodes" % n)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu = gpu
        self.rows = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 6 for k in range(4) if r[2 + k].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def load_fixture(L, p):
    path = os.path.join(ROOT, "tests", "golden", "size_fem2d_P1_L%d_p%g.npz" % (L, p))
    if not os.path.exists(path):
        return None, path
    return np.load(path, allow_pickle=False), path


def step_count_diff(its_a, fin_a, its_b, fin_b):
    """max over barrier steps of |Newton steps a - b|, the finalize pass (added into the last step) excluded; None if the
    t-schedules differ in length."""
    if its_a.shape != its_b.shape:
        return None
    ca, cb = its_a.sum(axis=0).astype(np.int64), its_b.sum(axis=0).astype(np.int64)
    ca[-1] -= fin_a
    cb[-1] -= fin_b
    return int(np.max(np.abs(ca - cb)))


def parity_record(sol, L, p, reduce_sum=None):
    """Timed solve vs the committed oracle fixture of the same workload.  reduce_sum: all-reduce (sum) of a float64 array
    over the ranks of a partitioned solve (sol["z"] then holds this rank's nodes, sol["node_range"] their global range)."""
    fx, path = load_fixture(L, p)
    S = sol["SOL_main"]
    rec = {"objective": float(S["c_dot_Dz"][-1]), "its_sum": int(S["its"].sum()), "its_finalize": int(S.get("its_finalize", 0))}
    if fx is None:
        rec["fixture"] = None
        return rec
    meta = json.loads(str(fx["meta"]))
    st = int(meta["stride"])
    z = sol["z"]
    i0 = sol["node_range"][0] if sol.get("node_range") else 0
    first = (-i0) % st                                      # first local node that the strided fixture holds
    zs = z[first::st]
    ref = fx["z"][(i0 + first) // st:(i0 + first) // st + zs.shape[0]]
    sums = np.array([float(np.sum((zs - ref) ** 2)), float(np.sum(ref ** 2)), float(np.sum(z ** 2))])
    if reduce_sum is not None:
        sums = reduce_sum(sums)
    rec.update({
        "fixture": os.path.relpath(path, ROOT), "oracle": "oracle/mgb_oracle.py via tests/golden/make_size_fixtures.py",
        "rel_vs_fixture": float(np.sqrt(sums[0] / sums[1])),
        "znorm_rel_vs_fixture": float(abs(np.sqrt(sums[2]) - float(fx["znorm"])) / float(fx["znorm"])),
        "objective_rel_vs_fixture": float(abs(rec["objective"] - float(fx["c_dot_Dz"][-1])) / abs(float(fx["c_dot_Dz"][-1]))),
        "its_sum_oracle": int(fx["its"].sum()), "its_finalize_oracle": int(fx["its_finalize"]),
        "barrier_steps": [int(S["its"].shape[1]), int(fx["its"].shape[1])],
        "max_step_count_diff_excl_finalize": step_count_diff(S["its"], rec["its_finalize"], fx["its"], int(fx["its_finalize"])),
    })
    rec["pass"] = bool(rec["rel_vs_fixture"] < 1e-6 and rec["objective_rel_vs_fixture"] < 1e-8 and
                       rec["max_step_count_diff_excl_finalize"] is not None and rec["max_step_count_diff_excl_finalize"] <= 1)
    return rec


def dump_outputs(out_dir, sol, budget=DUMP_BYTES):
    """Write what mgb_solve returned to its caller -- z and SOL_main without its wall-clock fields -- as float64 out_dir/<name>.npy.
    If the per-node arrays (z, z_unfinalized) do not fit in `budget` bytes, the same fixed sample of their rows (seed 0) is written
    instead, and the row numbers as node_rows.npy.  Returns the names written."""
    S = sol["SOL_main"]
    out = {k: np.asarray(S[k], dtype=np.float64) for k in ("its", "its_finalize", "ts", "kappas", "c_dot_Dz")}
    nodes = {"z": sol["z"], "z_unfinalized": S["z_unfinalized"]}
    n = sol["z"].shape[0]
    row_bytes = sum(8 * a[0].size for a in nodes.values())
    room = budget - sum(a.nbytes for a in out.values()) - 128 * (len(out) + len(nodes) + 1)     # 128: .npy header
    if n * row_bytes > room:
        rows = np.sort(np.random.default_rng(0).choice(n, room // (row_bytes + 8), replace=False))
        nodes = {k: a[rows] for k, a in nodes.items()}
        nodes["node_rows"] = rows
    out.update((k, np.asarray(a, dtype=np.float64)) for k, a in nodes.items())
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return sorted(out)


def oracle_solve(L, p):
    """ONE full-tolerance oracle solve; returns (value, seconds, Newton steps, n, objective)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import mgb_oracle as O
    prob = build_problem(L, p)
    t0 = time.time()
    sol = O.mgb_solve(prob)
    dt = time.time() - t0
    its = int(sol["SOL_main"]["its"].sum())
    n = prob.geometry.n
    return n * its / dt, dt, its, n, float(sol["SOL_main"]["c_dot_Dz"][-1])


def cpu_sample_text(L, n, p, its, dt):
    return ("CPU oracle (NumPy/SciPy SuperLU restatement of the reference path, 1 thread): ONE full-tolerance solve of %s, "
            "t-ramp to t >= 1/sqrt(eps) incl. finalize: %d Newton steps in %.1f s" % (workload_name(L, p, n), its, dt))


def reference_arm(args, rank, world):
    if rank != 0:
        return
    v, dt, its, n, obj = oracle_solve(args.ref_L, args.p)
    sample = cpu_sample_text(args.ref_L, n, args.p, its, dt)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": 1,
        "warmup": 0, "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.ref_L, args.p, n) + " -- the bounded sample of the headline workload (L=10, n=1572864) the CPU path "
                               "finishes in about two minutes; the GPU arm reports the same L in `same_config`",
                   "sample": sample, "objective": obj, "newton_steps": its,
                   "requested_steps_warmup": [args.steps, args.warmup],
                   "note": "deterministic CPU path: run once, not warmup+steps times"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference is Julia (absent here, baseline/run_reference.jl is its script); its CPU path is represented by the oracle port",
    }))


def fem3d_record(args, cfg, rank, world, local_rank, sharded, new_comm, barrier, tmax_over_ranks):
    """Sub-record on config C4's family: mgb_solve(assemble(amg(fem3d k=1 on c^3 hexahedra)); p=1; t=t0), ONE resident solve after one
    warm-up solve, elements partitioned over the ranks for N > 1 (strong scaling, like the headline record).  Parity for N > 1:
    rank 0 then solves the whole problem alone on its GPU and the objective / |z| are compared."""
    import torch
    from mgbx import geometry as G, hierarchy as H, native, problem as P, solver
    c = args.fem3d_c
    t0 = time.time()
    prob = P.assemble(H.amg(G.structured_box(3, c, k=1)), p=1.0)
    host_build_s = time.time() - t0
    n = prob.geometry.n
    bw = solver.barrier_weights(prob.M[0].w)
    if sharded:
        from mgbx import partition
        lprob = partition.shard_problem(prob, rank, world)
        lbw = partition.shard_barrier_weights(bw, *lprob.node_range)
    else:
        lprob, lbw = prob, bw
    h = native.Handle(lprob, barrier_weights=lbw, device=local_rank, comm=new_comm(), **cfg)
    try:
        for rep in range(2):
            h.set_grids(None, lprob.g)
            barrier()
            t1 = time.time()
            sol = solver.mgb_solve(lprob, handle=h, t=args.fem3d_t)
            barrier()
            dt = time.time() - t1
        info = h.solver_info()
    finally:
        h.close()
    dt = tmax_over_ranks(dt)
    S, st = sol["SOL_main"], sol["stats"]
    its = int(S["its"].sum())
    z2 = float(np.sum(sol["z"] ** 2))
    if sharded:
        t = torch.tensor([z2], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t)
        z2 = float(t.cpu()[0])
    rec = {"workload": "mgb_solve(assemble(amg(fem3d(k=1) on %d^3 hexahedra)); p=1.0; t=%g): n=%d broken nodes, fine unknowns %d"
                       % (c, args.fem3d_t, n, prob.M[0].R_fine[-1].shape[1]),
           "time_to_solution_s": dt, "value": n * its / dt, "unit": UNIT, "newton_steps": its, "barrier_steps": int(S["its"].shape[1]),
           "pcg_iters": int(st["pcg_iters"]), "solve_failures": int(st["solve_failures"]),
           "stage_ms": {k: st[k] for k in ("ms_f01", "ms_f2", "ms_solve")}, "objective": float(S["c_dot_Dz"][-1]), "znorm": float(np.sqrt(z2)),
           "host_build_s": host_build_s, "levels": info.get("m"), "row_sharded_levels": info.get("nshard", 0)}
    if sharded:
        if rank == 0:
            ref = solver.mgb_solve(prob, config=dict(device=local_rank, **cfg), t=args.fem3d_t)
            R = ref["SOL_main"]
            zr = float(np.linalg.norm(ref["z"]))
            rec["parity_vs_single_gpu"] = {
                "objective_rel_diff": float(abs(rec["objective"] - R["c_dot_Dz"][-1]) / abs(R["c_dot_Dz"][-1])),
                "znorm_rel_diff": float(abs(rec["znorm"] - zr) / zr), "newton_steps_single": int(R["its"].sum()),
                "barrier_steps_single": int(R["its"].shape[1]), "pcg_iters_single": int(ref["stats"]["pcg_iters"]),
                "single_gpu_e2e_s": float(ref["stats"]["create_s"] + sum(ref["stats"][k] for k in ("ms_f01", "ms_f2", "ms_solve")) * 1e-3)}
            pv = rec["parity_vs_single_gpu"]
            pv["pass"] = bool(pv["objective_rel_diff"] < 1e-8 and pv["znorm_rel_diff"] < 1e-6)
        barrier()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mgbx")
    ap.add_argument("--L", type=int, default=10, help="fem2d_P1 subdivision level (10: n = 1 572 864)")
    ap.add_argument("--p", type=float, default=1.5)
    ap.add_argument("--ref-L", type=int, default=REF_L)
    ap.add_argument("--cpu-L", type=int, default=CPU_L)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-same-config", action="store_true")
    ap.add_argument("--replicas", action="store_true", help="N > 1: N independent solves instead of one element-partitioned solve")
    ap.add_argument("--no-profile-pass", action="store_true")
    ap.add_argument("--fem3d-c", type=int, default=64, help="fem3d sub-record: k=1 hexahedra per edge (64: n = 2 097 152); 0 = skip")
    ap.add_argument("--fem3d-t", type=float, default=0.01, help="initial t of the fem3d sub-record (DESIGN.md: t = 0.1 stalls in the reference algorithm itself on >= 32^3)")
    ap.add_argument("--config", action="append", default=[], help="mgbx_config override key=value (repeatable)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed solve as DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and world > 1 and not args.replicas:
        ap.error("--dump-outputs needs the whole z on one rank: run on one GPU or with --replicas")

    sys.dont_write_bytecode = True
    if "NUMBA_CACHE_DIR" not in os.environ:
        os.environ["NUMBA_CACHE_DIR"] = tempfile.mkdtemp(prefix="mgbx-bench-numba-")
        atexit.register(shutil.rmtree, os.environ["NUMBA_CACHE_DIR"], True)

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    cfg = {}
    for kv in args.config:
        k, v = kv.split("=")
        cfg[k] = float(v) if ("." in v or "e" in v.lower()) else int(v)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libmgbx has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import mgbx  # noqa: F401
    from mgbx import native, solver

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_sum(a):
        if world == 1:
            return a
        t = torch.tensor(a, dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return t.cpu().numpy()

    prob = build_problem(args.L, args.p)
    n = prob.geometry.n
    bw = solver.barrier_weights(prob.M[0].w)
    sharded = world > 1 and not args.replicas
    comm_made = []

    def new_comm():
        """(rank, world, fresh NCCL id) for one handle: elements are partitioned over the ranks (partition.py)."""
        if not sharded:
            return None
        if comm_made:
            return (rank, world, None)             # later handles reuse the process-wide NCCL communicator
        uid = [native.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm_made.append(True)
        return (rank, world, uid[0])

    if sharded:
        from mgbx import partition
        lprob = partition.shard_problem(prob, rank, world)
        lbw = partition.shard_barrier_weights(bw, *lprob.node_range)
    else:
        lprob, lbw = prob, bw
    h = native.Handle(lprob, barrier_weights=lbw, device=local_rank, comm=new_comm(), **cfg)
    g0 = lprob.g

    def resident_step():
        h.set_grids(None, g0)                      # restart from the boundary data (device copy of 25 MB)
        sol = solver.mgb_solve(lprob, handle=h)
        return sol

    for _ in range(args.warmup):
        resident_step()

    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = h.launch_count()
    t0 = time.time()
    e0.record()
    for _ in range(args.steps):
        sol = resident_step()
    e1.record()
    barrier()
    wall = time.time() - t0
    dev_s = e0.elapsed_time(e1) * 1e-3
    launches = h.launch_count() - l0
    sampler.stop_flag = True
    its_total = int(sol["SOL_main"]["its"].sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sol)
    stats = sol["stats"]
    if sharded:
        sol["node_range"] = lprob.node_range
    parity = parity_record(sol, args.L, args.p, reduce_sum if sharded else None)

    # end-to-end through the public API with host buffers (handle creation + solve + z back), every step
    e2e_times = []
    h2d = 0
    for M in lprob.M[:1]:      # the feasibility AMG is only uploaded when phase I runs (it does not here)
        h2d += M.w.nbytes + sum(a.nbytes for a in M.geometry.operators.values())
        h2d += sum(R.data.nbytes + R.indices.nbytes * 2 + R.indptr.nbytes * 2 for R in M.R_fine[-1:])
        h2d += sum(T.data.nbytes + T.indices.nbytes * 2 + T.indptr.nbytes * 2 for T in M.T)
    h2d += lprob.f.nbytes + lprob.g.nbytes + sum(pc.A.nbytes + pc.b.nbytes for pc in lprob.Q.pieces)
    d2h = 2 * lprob.g.nbytes                              # z and z_unfinalized
    for k in range(1 + args.steps):      # one untimed warm-up call (first-use costs of a fresh handle), then the timed ones
        barrier()
        t1 = time.time()
        sol_e = solver.mgb_solve(prob, comm=new_comm(), config=dict(device=local_rank, **cfg))
        barrier()
        if k > 0:
            e2e_times.append(time.time() - t1)
        e2e_create = sol_e["stats"]["create_s"]
    its_e = int(sol_e["SOL_main"]["its"].sum())

    # profile pass: every kernel launch timed with CUDA events on the library's stream
    roof = None
    kstats = None
    if not args.no_profile_pass:
        h.set_profile(1)
        h.kernel_stats(reset=True)
        pstats = resident_step()["stats"]
        kstats = h.kernel_stats(reset=True)
        h.set_profile(0)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        counts = {k: v[0] for k, v in kstats.items()}
        ab = algorithmic_bytes(lprob, h, counts)
        info = h.solver_info()
        total_ms = max(1e-9, sum(v[1] for v in kstats.values()))

        try:
            ncu_tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except Exception:
            ncu_tr = {}
        gen = int(h.cfg.persistent)

        def traffic(cls, nl):
            """DRAM bytes per launch from a committed `ncu --set full` capture of the SAME kernel on this workload (never
            measured in this run: ncu numbers cannot be taken inside a timed bench).  Returns (bytes, source) or (None, why)."""
            key = {"elem_f01": "k_elem_f01", "elem_f2": "k_elem_f2", "pcg_persistent": "k_pcg2" if gen == 2 else "k_pcg_persistent"}.get(cls)
            e = ncu_tr.get(key)
            if e is None:
                return None, "no committed ncu capture of %s" % key
            src = "committed ncu --set full capture %s (%s)" % (e.get("capture", "?"), e.get("build", "build not recorded"))
            if cls == "pcg_persistent":
                return 1e6 * e["dram_mb_per_launch"] / e["pcg_iterations_in_launch"] * pstats["pcg_iters"] / nl, src + ", scaled by PCG iterations"
            return 1e6 * e["dram_mb_per_launch"], src

        def line(cls):
            nl, ms = kstats[cls]
            if not nl:
                return None
            if cls == "pcg_persistent":
                # one launch = one whole PCG solve; bytes = iterations of the profiled solve x bytes per iteration
                bpl = ab.get("pcg_iteration", 0) * pstats["pcg_iters"] / nl
            else:
                bpl = ab.get(cls)
            ach = bpl / (ms * 1e-3 / nl) / 1e9 if bpl else None
            tr, tr_src = traffic(cls, nl)
            return {"bound": "hbm", "kernel": cls, "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": (ach / peak) if ach else None, "traffic": tr, "traffic_source": tr_src,
                    "algorithmic_bytes_per_launch": bpl, "launches": nl, "avg_launch_us": 1e3 * ms / nl,
                    "share_of_device_time": ms / total_ms}
        dom = max(kstats, key=lambda k: kstats[k][1])
        roof = line(dom)
        roof["peak_source"] = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s"
        if dom == "pcg_persistent":
            roof["note"] = ("one launch = one whole V-cycle-PCG solve (%d levels: %s unknowns, %.1f PCG iterations per launch); its working set "
                            "(matrices + vectors of all levels, ~%.0f MB) is L2-resident, so the HBM peak is a reference line, not a ceiling; "
                            "the kernel is bound by grid-barrier and dependent-load latency (see DESIGN.md)"
                            % (info["nlev"], info["m"], pstats["pcg_iters"] / max(1, kstats[dom][0]), sum(12 * z for z in info["nnz"]) / 1e6))
        roof_all = {c: line(c) for c in ("elem_f01", "elem_f2", "elem_generic_f01", "elem_generic_f2", "csr_gather", "spgemm", "pcg_persistent")
                    if kstats.get(c, (0, 0))[0]}
    h.close()

    # the same GPU path at the levels the CPU arms run: like-for-like pairs for cpu_baseline / --impl reference
    same = None
    if world == 1 and not args.no_same_config:
        same = {}
        for Ls in sorted({args.cpu_L, args.ref_L}):
            ps = build_problem(Ls, args.p)
            hs = native.Handle(ps, barrier_weights=solver.barrier_weights(ps.M[0].w), device=local_rank, **cfg)
            try:
                for rep in range(3):
                    hs.set_grids(None, ps.g)
                    torch.cuda.synchronize()
                    t1 = time.time()
                    ss = solver.mgb_solve(ps, handle=hs)
                    torch.cuda.synchronize()
                    dts = time.time() - t1
            finally:
                hs.close()
            t1 = time.time()
            se = solver.mgb_solve(ps, config=dict(device=local_rank, **cfg))
            dte = time.time() - t1
            its_s = int(ss["SOL_main"]["its"].sum())
            same["L%d" % Ls] = {"workload": workload_name(Ls, args.p, ps.geometry.n), "newton_steps": its_s, "s_per_solve_resident": dts,
                                "value": ps.geometry.n * its_s / dts, "e2e_s": dte, "e2e_value": ps.geometry.n * int(se["SOL_main"]["its"].sum()) / dte,
                                "parity": parity_record(ss, Ls, args.p)}

    def tmax_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.cpu()[0])

    # N > 1: the partitioned solve against the single-GPU solve of the same problem (rank 0 solves it alone)
    vs_single = None
    if sharded:
        zz = reduce_sum(np.array([float(np.sum(sol["z"] ** 2))]))
        if rank == 0:
            ref1 = solver.mgb_solve(prob, config=dict(device=local_rank, **cfg))
            R1 = ref1["SOL_main"]
            zr = float(np.linalg.norm(ref1["z"]))
            vs_single = {"objective_rel_diff": float(abs(sol["SOL_main"]["c_dot_Dz"][-1] - R1["c_dot_Dz"][-1]) / abs(R1["c_dot_Dz"][-1])),
                         "znorm_rel_diff": float(abs(np.sqrt(zz[0]) - zr) / zr), "newton_steps_single": int(R1["its"].sum()),
                         "same_t_schedule": bool(R1["ts"].shape == sol["SOL_main"]["ts"].shape and np.allclose(R1["ts"], sol["SOL_main"]["ts"], rtol=1e-12))}
            vs_single["pass"] = bool(vs_single["objective_rel_diff"] < 1e-8 and vs_single["znorm_rel_diff"] < 1e-6)
        barrier()
    parity["vs_single_gpu"] = vs_single

    # everything the headline record needs is reduced BEFORE the fem3d sub-record runs, so that nothing the sub-record does
    # (it exercises the row-sharded solve for N >= 4) can take the headline line down with it
    tmax = torch.tensor([dev_s, wall, float(np.mean(e2e_times))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dev_s, wall, e2e_s = [float(x) for x in tmax.cpu()]

    fem3d = None
    if args.fem3d_c > 0:
        try:
            fem3d = fem3d_record(args, cfg, rank, world, local_rank, sharded, new_comm, barrier, tmax_over_ranks)
        except BaseException as e:     # the sub-record must never take the headline line down with it
            fem3d = {"error": repr(e)[:300]}
    nshard = int(info.get("nshard", 0)) if (roof is not None) else 0
    units = 1 if sharded else world       # sharded: ONE solve split over the ranks; replicas: one solve per rank
    value = units * n * its_total * args.steps / dev_s
    e2e_value = units * n * its_e / e2e_s

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.L, args.p, n) + ", nu=2, nD=4, fine unknowns %d" % prob.M[0].R_fine[-1].shape[1],
                   "newton_steps_per_solve": its_total, "time_to_solution_s": dev_s / args.steps,
                   "parallelism": ("1 GPU" if world == 1 else
                                   ("element partition over %d GPUs: barrier / gradient / Hessian kernels sharded by element block, NCCL all-reduce "
                                    "of R'g, Hessian values and scalars; multigrid-PCG solve %s (strong scaling: ONE solve)"
                                    % (world, ("row-sharded over the ranks inside the persistent kernel on its %d leading level(s) (peer stores over NVLink into "
                                               "CUDA-IPC exchange arenas, cross-GPU flag barrier), replicated below" % nshard) if nshard else "replicated on every rank"))
                                   if sharded else "replicas: %d independent solves, no data-path collective" % world),
                   "l2_policy": "working set (>= 600 MB of grids, operators and CSR values) exceeds the 126 MB L2; no flush needed",
                   "wall_s_timed_region": wall, "mgbx_config_overrides": cfg},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d) * (world if sharded else 1), "d2h_bytes_per_step": int(d2h) * (world if sharded else 1),
                "s_per_step": e2e_s, "create_s": e2e_create,
                "includes": "handle creation (layout conversion + H2D), plan build, solve, z and z_unfinalized D2H"},
        "parity": parity,
        "gpu_launches": int(launches),
        "stage_ms_per_solve": {k: stats[k] for k in ("ms_f01", "ms_f2", "ms_solve")},
        "counts_per_solve": {k: stats[k] for k in ("f01_evals", "f2_evals", "linear_solves", "pcg_iters", "solve_failures")},
        "clocks": sampler.summary(),
    }
    if roof:
        out["roofline"] = roof
        out["roofline_by_kernel"] = {k: {kk: v[kk] for kk in ("achieved", "frac", "traffic", "traffic_source", "avg_launch_us", "share_of_device_time", "algorithmic_bytes_per_launch")}
                                     for k, v in roof_all.items() if v}
        out["solver_plan"] = info
        out["kernel_classes"] = {k: {"launches": v[0], "ms": round(v[1], 3)} for k, v in kstats.items()}
    if same:
        out["same_config"] = same
    if fem3d:
        out["fem3d"] = fem3d
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, its, nn, obj = oracle_solve(args.cpu_L, args.p)
        out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": cpu_sample_text(args.cpu_L, nn, args.p, its, dt),
                               "same_config_gpu": "same_config.L%d" % args.cpu_L}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


def algorithmic_bytes(prob, h, counts):
    """Algorithmic bytes PER LAUNCH of each kernel class at the fine level (SURVEY.md section 8d, DESIGN.md section 4).
    counts: {class: launches} of the profiled solve, used to spread per-assembly totals over a class's launches."""
    M = prob.M[0]
    n, N, p = M.geometry.n, M.geometry.N, M.geometry.V
    nD, nu = M.nD, M.nu
    nops = len({op for (_, op) in M.D if op != "id"})
    info = h.solver_info()
    nE = 1 if info["condensed"] else 0            # default problem: the :full slack is eliminated node-locally
    nK = nD - nE
    pairs = (nu - nE) ** 2
    ops_b = nops * p * p * N
    out = {}
    # fused element kernels: zf (nu), f grid (nD), w, operator blocks once; write gb (nu)  /  hEEinv, hKE, Hblk
    out["elem_f01"] = 8 * (n * (nu + nD + 1) + ops_b + nu * n)
    out["elem_f2"] = 8 * (n * nu + ops_b + n * (nE * (nE + 1) // 2 + nK * nE) + pairs * N * p * p)
    out["elem_generic_f01"] = out["elem_f01"]
    out["elem_generic_f2"] = 8 * (n * nu + ops_b + nu * nu * N * p * p)      # coarse-level systems: nothing eliminated, nu^2 block pairs
    out["node_f01"] = 8 * (n * (nu + nD + 1 + nD) + ops_b)
    out["node_f2"] = 8 * (n * (nu + nK * (nK + 1) // 2 + nE * (nE + 1) // 2 + nK * nE) + ops_b)
    out["blockgrad"] = 8 * (n * nD + ops_b + nu * n)
    out["blockhess"] = 8 * (n * nK * (nK + 1) // 2 + ops_b + pairs * N * p * p)
    if info["nlev"]:
        nnz0 = info["nnz"][0]
        out["csr_gather"] = 8 * info["hblk_entries"] + 4 * info["assembly_terms"] + 8 * nnz0 + nnz0 // 2
        # all Galerkin gathers of one assembly, spread over the class's launches per assembly
        tot = 12 * info["galerkin_terms"] + 8 * sum(info["nnz"][1:]) * 2
        if counts.get("spgemm") and counts.get("elem_f2"):
            out["spgemm"] = tot / (counts["spgemm"] / counts["elem_f2"])
        out["pcg_iteration"] = pcg_iteration_bytes(info)
    return out


def pcg_iteration_bytes(info, nu_sweeps=2):
    """One PCG iteration of the persistent kernel, with SURVEY.md section 8(d)'s SpMV figure `12 nnz + 20 rows` per pass:
    per non-bottom level 1 fused pre-smoothing pass + 1 residual + nu post passes over A, one pass over T and T' each; the PCG
    mat-vec on the top level; 5 vector streams of the PCG update."""
    b = 0
    L = info["nlev"]
    for q in range(L):
        m, nnz, nnzT = info["m"][q], info["nnz"][q], info["nnzT"][q]
        if q == L - 1:
            b += 8 * m * m if info["bottom_dense"] else 30 * (12 * nnz + 20 * m)
            continue
        b += (2 + nu_sweeps) * (12 * nnz + 20 * m) + (12 * nnzT + 20 * m) + (12 * nnzT + 20 * info["m"][q + 1])
    b += 12 * info["nnz"][0] + 20 * info["m"][0] + 5 * 8 * info["m"][0]
    return b


if __name__ == "__main__":
    main()
