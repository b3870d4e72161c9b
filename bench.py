#!/usr/bin/env python
"""bench.py -- 3D swelling (swelling-3d.py) solve phase on B200: time-to-1e-8, GMRES iteration
throughput, SpMV HBM roofline.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--mesh-n M] [--dump-outputs DIR]

A "step" is ONE complete `Solver.solve(b, x)` of the assembled three-field system from a zero
initial guess to relative residual 1e-8 (right-preconditioned GMRES + block `diagonal`
preconditioner: one SA-AMG V-cycle on the solid block, one on the fluid-velocity block, and the additive
Cahouet-Chabard pressure Schur preconditioner: one V-cycle on the lumped-mass Schur complement + Chebyshev(4) on the pressure mass matrix) -- set-up (assembly, upload,
AMG hierarchy) is outside the timed region exactly as the reference times only `ksp.solve`
(lib/Solver.py:148-152).  `value` = DoFs solved to 1e-8 per second = n_dofs / time-to-1e-8 over the K
timed steps (whole job, all ranks; a weaker preconditioner that needs more iterations scores LOWER);
`e2e` is the same through the host-buffer entry point (poro_ksp_solve_host: b copied H2D and x copied
D2H inside the timed region).  Iteration throughput, phase profile and the roofline of the dominant kernel
are measured in a SEPARATE profiled pass after the timed ones.

`--dump-outputs DIR` writes what the last timed step returned to its caller, as float64 .npy files: `x` (the solution,
`x_rank<r>` per rank when several ranks share the mesh) and `residual_history` (the outer KSP's residual norms).  The
inputs depend only on the arguments, so two builds run with the same arguments can be compared file by file.

Weak scaling: N GPUs solve the cube with ~N x the DoFs of the 1-GPU mesh, row-partitioned in
z-slabs (one rank per GPU, NCCL halo exchange + all-reduce).

`--impl reference`: the reference's own stack (petsc4py/dolfin/hypre) is absent from this image
and unbuildable offline, so the reference arm times the CPU oracle port (numpy/scipy set-up + C/OpenMP solve
loop restating the same algorithm, oracle/) on the host cores, on the SAME mesh as the GPU arm at that N.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("PORO_LOG_STDERR", "1")      # stdout carries only the JSON line

BENCH_OPTIONS = """
-global_ksp_type gmres
-global_ksp_pc_side right
-global_ksp_gmres_verify_true_residual 1
-s_ksp_type preonly
-s_pc_type hypre
-s_pc_amg_theta 0.04
-s_pc_amg_coarse_size 6000
-poro_amg_dense_limit 8192
-fp_ksp_type preonly
-fp_pc_fieldsplit_type schur
-fp_pc_fieldsplit_schur_fact_type lower
-fp_pc_fieldsplit_schur_precondition cc
-fp_pc_fieldsplit_order fp
-fp_fieldsplit_0_ksp_type preonly
-fp_fieldsplit_0_pc_type hypre
-fp_fieldsplit_0_pc_amg_theta 0.04
-fp_fieldsplit_0_pc_amg_coarse_size 6000
-fp_fieldsplit_1_ksp_type preonly
-fp_fieldsplit_1_pc_type hypre
-fp_fieldsplit_1_pc_amg_coarse_size 6000
"""
# `-fp_pc_fieldsplit_schur_precondition cc`: the additive Cahouet-Chabard form of the pressure Schur preconditioner -- the pressure
# treatment of the reference's 3-way variants (beta_CC1 / beta_CC2, lib/Assembler.py:131-137) inside the 2-way fieldsplit -- with a
# V-cycle on the velocity block.  PETSc's `selfp` (the set benchmarked until the middle of round 2, kept below and parity-tested)
# loses mesh independence once the viscous part of P_ff overtakes its mass + drag part: 36 / 44 / 55 / 70 / 109 iterations at
# N = 34 / 43 / 54 / 68 / 101 against 27 / 29 / ... with `cc` (profiles/r2_schur_cc.md).
BENCH_OPTIONS_SELFP = (BENCH_OPTIONS.replace("-fp_pc_fieldsplit_schur_precondition cc", "-fp_pc_fieldsplit_schur_precondition selfp")
                       .replace("-fp_fieldsplit_0_pc_type hypre\n-fp_fieldsplit_0_pc_amg_theta 0.04\n-fp_fieldsplit_0_pc_amg_coarse_size 6000\n",
                                "-fp_fieldsplit_0_pc_type chebyshev\n"))
BENCH_OPTIONS_CC = BENCH_OPTIONS
PHASE_NAMES = {0: "outer_A_apply", 1: "pc_apply", 2: "s_solve", 3: "fp_split0(f)", 4: "fp_split1(p)", 5: "gram_schmidt",
               6: "fp_coupling", **{8 + l: "s_amg_L%d" % l for l in range(8)}, **{16 + l: "f_amg_L%d" % l for l in range(8)},
               **{24 + l: "p_amg_L%d" % l for l in range(8)}, 32: "A_remainder_csr", 33: "A_part0", 34: "A_part1", 35: "A_part2", 36: "A_part3",
               37: "s_L0_cheby_step_launch"}
RTOL = 1e-8
METRIC = "3D swelling (swelling-3d.py) solve to rtol 1e-8: DoFs solved per second (n_dofs / time-to-1e-8)"
UNIT = "DoF/s"
DUMP_BYTES = 64 * 10 ** 6        # --dump-outputs writes at most this much in all (all ranks together)


def dump_outputs(out_dir: str, arrays: dict, budget: int) -> None:
    """Writes each array as out_dir/<name>.npy in float64, in at most `budget` bytes.  Smaller arrays are written whole first; an
    array that does not fit its share of what is left is replaced by the entries at a fixed sample of indices (seed 0, ascending
    order), the same sample in every run with the same arguments."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: np.size(kv[1]))
    for i, (name, a) in enumerate(items):
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        cap = (budget // (len(items) - i) - 128) // a.itemsize     # 128 B: the .npy header
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        budget -= os.path.getsize(path)


def active_options() -> str:
    """The option text of this run: BENCH_OPTIONS plus the A/B switches of PORO_EXTRA_OPTIONS (later keys win)."""
    extra = os.environ.get("PORO_EXTRA_OPTIONS", "").strip()
    return BENCH_OPTIONS + ("\n" + extra.replace(";", "\n") + "\n" if extra else "")


def mesh_for_gpus(base_n: int, gpus: int) -> int:
    """Weak scaling: cube side so that DoFs ~ gpus x DoFs(base_n)."""
    return int(round(base_n * gpus ** (1.0 / 3.0)))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi SM clocks and throttle reasons during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device: int):
        self.device, self.samples, self.stop_flag, self.th = device, [], False, None

    def _run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm)}


def oracle_solver(sys_, par, max_it, options_text=None):
    """The CPU port of the benchmarked algorithm (same options as BENCH_OPTIONS, or as `options_text`: the selfp / cc
    Schur preconditioner and the Chebyshev / V-cycle choice on the velocity block are read from it).

    Returns {label: (run, cores)}: the numpy/scipy oracle on one thread, and the same preconditioner handed
    to the C + OpenMP solve loop (oracle/csrc/cpu_solver.c) with the thread count that is fastest on this host."""
    from oracle.amg import SAAMG, rigid_body_modes
    from oracle.blockpc import BlockPC, SchurLower, SchurLowerCC, cc_from_matrices, krylov_solver
    from oracle.krylov import gmres
    from oracle import cport
    opts = {}
    for line in (options_text if options_text is not None else active_options()).splitlines():
        w = line.split()
        if w and not w[0].startswith("#"):
            opts[w[0].lstrip("-")] = w[-1] if len(w) > 1 else None
    dim = sys_.dim
    B = rigid_body_modes(sys_.coords_s, dim)
    # coarsening stops below 6 000 (global) rows, where one dense inverse is cheaper than further latency-bound levels
    amg_s = lambda M: SAAMG(M, dim, B, theta=0.04, coarse_size=6000, dense_limit=8192)   # -s_pc_amg_theta 0.04 -s_pc_amg_coarse_size 6000
    cheb_f = lambda M: SAAMG(M, dim, B, max_levels=1, cheby_degree=4, dense_limit=0)   # -fp_fieldsplit_0_pc_type chebyshev
    amg_p = lambda M: SAAMG(M, 1, None, coarse_size=6000, dense_limit=8192)
    k_f = cheb_f
    if opts.get("fp_fieldsplit_0_pc_type", "chebyshev") != "chebyshev":
        # -fp_fieldsplit_0_pc_type hypre -fp_fieldsplit_0_pc_amg_theta .. -fp_fieldsplit_0_pc_amg_coarse_size ..
        k_f = lambda M: SAAMG(M, dim, B, theta=float(opts.get("fp_fieldsplit_0_pc_amg_theta", 0.08)),
                              coarse_size=int(opts.get("fp_fieldsplit_0_pc_amg_coarse_size", 400)), dense_limit=8192)
    if opts.get("fp_pc_fieldsplit_schur_precondition", "selfp") == "cc":
        d_mass, S_visc = cc_from_matrices(sys_, par)
        cheb_p = lambda M: SAAMG(M, 1, None, max_levels=1, cheby_degree=4, dense_limit=0)
        mkfp = lambda M: SchurLowerCC(M, sys_.nf, sys_.np_, krylov_solver("preonly", k_f), krylov_solver("preonly", amg_p),
                                      krylov_solver("preonly", cheb_p), d_mass, S_visc)
    else:
        mkfp = lambda M: SchurLower(M, sys_.nf, sys_.np_, krylov_solver("preonly", k_f), krylov_solver("preonly", amg_p), "f")
    # the two vector hierarchies are independent: build them side by side (scipy's sparse kernels release the GIL) and hand the
    # finished objects to the factories when BlockPC asks for exactly these blocks
    from concurrent.futures import ThreadPoolExecutor
    from oracle.blockpc import submatrix
    pre = {}
    if k_f is not cheb_f:
        Ms, Mf = submatrix(sys_.P, sys_.is_s, sys_.is_s), submatrix(sys_.P, sys_.is_f, sys_.is_f)
        with ThreadPoolExecutor(2) as ex:
            fs, ff = ex.submit(amg_s, Ms), ex.submit(k_f, Mf)
            pre = {"s": (Ms, fs.result()), "f": (Mf, ff.result())}

    def prebuilt(key, make):
        def mk(M):
            if key in pre:
                M0, h = pre[key]
                if M0.shape == M.shape and M0.nnz == M.nnz and np.array_equal(M0.indices, M.indices) and np.array_equal(M0.data, M.data):
                    return h
            return make(M)
        return mk

    amg_s, k_f = prebuilt("s", amg_s), prebuilt("f", k_f)
    if opts.get("fp_pc_fieldsplit_schur_precondition", "selfp") == "cc":
        mkfp = lambda M: SchurLowerCC(M, sys_.nf, sys_.np_, krylov_solver("preonly", k_f), krylov_solver("preonly", amg_p),
                                      krylov_solver("preonly", cheb_p), d_mass, S_visc)
    else:
        mkfp = lambda M: SchurLower(M, sys_.nf, sys_.np_, krylov_solver("preonly", k_f), krylov_solver("preonly", amg_p), "f")
    pc = BlockPC(sys_, {"s": krylov_solver("preonly", amg_s), "fp": mkfp})
    A = sys_.A

    def run_numpy():
        return gmres(lambda v: A @ v, sys_.b, pc, rtol=RTOL, atol=0.0, dtol=1e20, max_it=max_it, restart=max(max_it, 1),
                     pc_side="right")

    out = {"numpy/scipy, 1 thread": (run_numpy, 1)}
    try:
        cs = cport.CSolver(sys_, pc)
        # thread count: hosts differ (shared vCPUs make a full OpenMP team slower than two threads), so probe
        # a few team sizes on a 4-iteration solve and keep the fastest
        tmax = max(cport.threads(), os.cpu_count() or 1)     # torchrun exports OMP_NUM_THREADS=1: size the team ourselves
        # (largest team first, halving while that does not make it slower: two probes on a healthy host)
        best_t, best_dt = 1, None
        for t in sorted({t for t in (1, 2, 4, 8, 16, 32, 64, tmax) if t <= tmax}, reverse=True):
            cport.set_threads(t)
            cs.solve(sys_.b, RTOL, 0.0, 1)
            t0 = time.perf_counter()
            cs.solve(sys_.b, RTOL, 0.0, 3)
            dt = time.perf_counter() - t0
            if best_dt is None or dt < best_dt:
                best_t, best_dt = t, dt
            elif dt > 1.25 * best_dt:
                break
        cport.set_threads(best_t)

        def run_c():
            return cs.solve(sys_.b, RTOL, 0.0, max_it)

        out["C + OpenMP solve loop on %d threads" % best_t] = (run_c, best_t)
    except Exception as e:                      # the C port is optional: report the numpy build alone
        print("[bench] C port of the CPU baseline unavailable: %r" % (e,), file=sys.stderr)
    return out


def cpu_baseline(mesh_n: int, x_gpu=None):
    """Oracle port timed on the host cores on the SAME mesh as the GPU arm: ONE full solve to rtol 1e-8 with the C + OpenMP
    solve loop (the bounded sample: about 5-15 s of CPU work after an untimed numpy set-up), its iteration count and the
    relative difference of its solution to the GPU's."""
    from oracle.problems import swelling
    sys_, par = swelling(3, mesh_n, "diagonal")
    runs = oracle_solver(sys_, par, 100)
    label = [k for k in runs if k.startswith("C + OpenMP")]
    label = label[0] if label else list(runs)[0]
    run, cores = runs[label]
    t0 = time.perf_counter()
    r = run()
    dt = time.perf_counter() - t0
    out = {"value": sys_.n / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": "same mesh N=%d (%d DoFs), one full solve to rtol 1e-8: %d its in %.2f s; %s; NOT PETSc/hypre"
                     % (mesh_n, sys_.n, r.its, dt, label),
           "its": int(r.its), "seconds": dt, "same_config": True,
           "true_rel_residual": float(np.linalg.norm(sys_.b - sys_.A @ r.x) / np.linalg.norm(sys_.b))}
    if x_gpu is not None and len(x_gpu) == len(r.x):
        out["rel_diff_x_gpu_vs_cpu"] = float(np.linalg.norm(x_gpu - r.x) / np.linalg.norm(r.x))
    return out


def run_reference(args):
    """The reference arm: the oracle port's solve of the SAME mesh the GPU arm solves at this N, on all host cores.
    Each step is one full solve."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    from oracle.problems import swelling
    N_arm = args.total_mesh_n or mesh_for_gpus(args.mesh_n, max(world, args.gpus))
    N = N_arm
    same = True
    if N > args.cpu_max_n:
        # the numpy set-up of the port does not fit the time budget on the weak-scaled mesh: the bounded sample is the
        # per-GPU share of the workload (the 1-GPU mesh).  DoF/s on the smaller mesh is an UPPER bound for the port's DoF/s on
        # the larger one (the iteration count grows with the mesh), i.e. the comparison errs in the CPU's favour.
        N = min(args.mesh_n, args.cpu_max_n)
        same = False
    sys_, par = swelling(3, N, "diagonal")
    runs = oracle_solver(sys_, par, 100)
    label = [k for k in runs if k.startswith("C + OpenMP")]
    label = label[0] if label else list(runs)[0]
    run, ncores = runs[label]
    run()                                           # warm-up solve
    for _ in range(max(0, min(args.warmup, 1) - 1)):
        run()
    t0 = time.perf_counter()
    its = 0
    for _ in range(args.steps):
        r = run()
        its += r.its
    dt = (time.perf_counter() - t0) / args.steps
    val = sys_.n / dt
    res = float(np.linalg.norm(sys_.b - sys_.A @ r.x) / np.linalg.norm(sys_.b))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "steps_timed": args.steps,
            "config": {"workload": workload_text(N, sys_.n, sys_.A.nnz, 100, "maxiter", 1), "same_config_as_gpu_arm": same,
                       "gpu_arm_mesh_n": N_arm,
                       "note": "CPU oracle port (numpy set-up + C/OpenMP solve loop), NOT PETSc/hypre; each step = one full "
                               "solve%s" % ("" if same else "; sample = the 1-GPU mesh (per-GPU share of the weak-scaled "
                                            "workload): the port's set-up of the N=%d mesh does not fit the time budget" % N_arm)},
            "time_to_1e-8_s": dt, "its_per_solve": its / args.steps, "true_rel_residual": res,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": ncores, "kind": "port",
                             "sample": "mesh N=%d (%d DoFs), %d full solves, %s; NOT PETSc/hypre" % (N, sys_.n, args.steps, label)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"x": r.x, "residual_history": r.history}, DUMP_BYTES)
    print(json.dumps(line))


def workload_text(N, n_global, nnzA, maxiter, restart, world):
    return ("swelling-3d.py -N %d (%d DoFs, nnz(A)=%d on rank 0), GMRES(right, maxiter=%d, restart=%s) + block 'diagonal' 2-way PC: "
            "SA-AMG V-cycle (s), SA-AMG V-cycle (f), additive Cahouet-Chabard pressure Schur preconditioner (V-cycle on P_pp - P_pf "
            "diag(c M_v)^-1 P_fp + Chebyshev(4) on the pressure mass matrix); rtol 1e-8, zero initial guess"
            % (N, n_global, nnzA, maxiter, restart))


def measured_traffic(kernel_key: str, bytes_per_launch: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    export (profiles/r2_ncu_traffic.json, written by profiles/ncu_traffic.py from the .ncu-rep of this round).  null when
    no capture of this kernel on a matrix of this size is committed."""
    p = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if not os.path.exists(p):
        return None, "no committed ncu capture"
    try:
        for e in json.load(open(p)).get("kernels", []):
            if e.get("key") == kernel_key and abs(e.get("algorithmic_bytes", 0) - bytes_per_launch) <= 0.02 * bytes_per_launch:
                return float(e["dram_bytes"]), e.get("source", p)
    except Exception as ex:
        return None, "unreadable: %r" % (ex,)
    return None, "no capture of this kernel at this size"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--mesh-n", type=int, default=34, help="cells per side at 1 GPU (swelling-3d.py -N)")
    ap.add_argument("--maxiter", type=int, default=100, help="solver maxiter = GMRES restart (swelling-3d.py:66: 100)")
    ap.add_argument("--total-mesh-n", type=int, default=0, help="cells per side of the WHOLE mesh at this GPU count (overrides the weak-scaling "
                    "rule; e.g. 101 = BASELINE config 5, 51.3 M DoFs)")
    ap.add_argument("--cpu-sample-n", type=int, default=0, help="(unused since round 2: the CPU arm runs the GPU arm's own mesh)")
    ap.add_argument("--cpu-max-n", type=int, default=40, help="largest mesh the CPU oracle port is set up for")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--assemble", default="device", choices=["device", "host"],
                    help="device: each rank generates its slab of A, P in HBM (csrc/gen.cu); host: hostfem element assembly + upload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (solution, residual history) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    from poro_b200.lib.backend import DeviceMatrix, DeviceVector, get_context
    from poro_b200.lib.IndexSet import IndexSet
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    from poro_b200.lib.Solver import Solver

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = get_context(local_rank)
    load_petsc_options(ctx, BENCH_OPTIONS, is_text=True)
    extra = os.environ.get("PORO_EXTRA_OPTIONS", "").strip()        # A/B switches of library tunables (e.g. "-poro_bsr_tma 0")
    if extra:
        load_petsc_options(ctx, extra.replace(";", "\n"), is_text=True)

    # ---- set-up (untimed): generate (or assemble) the system, build the preconditioner
    t_asm = time.perf_counter()
    N = args.total_mesh_n or mesh_for_gpus(args.mesh_n, world)
    gen_sys = None
    if args.assemble == "device":
        from poro_b200.generator import generate_swelling3d
        gen_sys = generate_swelling3d(ctx, N, "diagonal", rank, world)
        par, n_global = gen_sys.par, gen_sys.n_global
        b_np, bcs_p = gen_sys.b, gen_sys.bcs_sub_pressure
    elif world > 1:
        from poro_b200.partition import distributed_problem
        prob = distributed_problem(3, N, "diagonal", rank, world, ctx)
        sys_, par, n_global = prob.sys, prob.par, prob.n_global
        b_np, bcs_p = sys_.b, sys_.bcs_sub_pressure
    else:
        from hostfem.problems import swelling     # host-side input generation standing in for FEniCS assembly (not the oracle)
        sys_, par = swelling(3, N, "diagonal")
        n_global = sys_.n
        b_np, bcs_p = sys_.b, sys_.bcs_sub_pressure
    ctx.sync()
    t_asm = time.perf_counter() - t_asm
    par = dict(par)
    # swelling-3d.py:66: maxiter (= restart, lib/Solver.py:99-100) 100, at every N: the distributed hierarchies
    # (csrc/distamg.cu) keep the iteration count of the single-GPU solve
    maxiter = args.maxiter
    par.update({"solver rtol": RTOL, "solver atol": 0.0, "solver maxiter": maxiter, "solver type": "gmres"})
    t_set = time.perf_counter()
    if gen_sys is not None:
        imap = gen_sys.index_set()
        dA, dP = gen_sys.A, gen_sys.P
        nnzA = gen_sys.A.nnz
    else:
        imap = IndexSet(sys_.is_s, sys_.is_f, sys_.is_p, two_way=True, block_dim=3, coords_s=sys_.coords_s,
                        coords_p=sys_.coords_p) if world == 1 else prob.index_set()
        dA, dP = DeviceMatrix(sys_.A, ctx), DeviceMatrix(sys_.P, ctx)
        nnzA = sys_.A.nnz
    b_host = torch.from_numpy(np.ascontiguousarray(b_np)).pin_memory()
    x_host = torch.zeros_like(b_host).pin_memory()
    db = DeviceVector(b_np, ctx=ctx)
    dx = DeviceVector(n=len(b_np), ctx=ctx)
    pcw = Preconditioner(imap, dA, dP, None, par, bcs_p)
    pc = pcw.get_pc()
    solver = Solver(dA, db, pc, par, imap)
    solver.create_solver(dA, db, pc)
    ksp = solver.solver
    ctx.sync()
    t_set = time.perf_counter() - t_set

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    wall = {}

    def timed(fn, steps, tag="dev"):
        """K steps between barrier + synchronize; time = CUDA events on the library's stream, max over ranks."""
        barrier()
        t0 = time.perf_counter()
        ctx.timer_start()
        its = 0
        for _ in range(steps):
            its += fn()
        dt = ctx.timer_stop() / 1e3
        barrier()
        wall[tag] = time.perf_counter() - t0
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([dt, wall[tag]], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt, wall[tag] = float(t[0]), float(t[1])
        return dt, its

    def step_dev():
        ksp.solve(db, dx)
        return ksp.its

    def step_host():
        ksp.solve_host(b_host, x_host)
        return ksp.its

    for _ in range(args.warmup):
        step_dev()
    # ---- timed passes: NO profiler events, nothing but the solves between the barriers
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count()
    dt, its = timed(step_dev, args.steps)
    launches = ctx.launch_count() - l0
    reason, rnorm = ksp.reason, ksp.rnorm
    xs = dx.numpy()
    history = ksp.getConvergenceHistory()
    step_host()
    dt_e, its_e = timed(step_host, args.steps, "e2e")
    clocks = sampler.stop()
    # ---- separate profiled pass (CUDA events around phases and around every launch of the outer operator)
    prof_steps = max(1, min(args.steps, 3))
    ksp.profile(1)
    ctx.profile(1)
    dt_p, _ = timed(step_dev, prof_steps, "prof")
    op_ms, op_calls, op_bytes = ksp.profile(0)
    phases = ctx.profile(0)

    # ---- verification of the timed result (outside the timed region): true residual on every N
    dy = DeviceVector(n=len(b_np), ctx=ctx)
    dA.mult(dx, dy)                                   # raw-ordering operator incl. halo exchange (poro_mat_mult)
    ctx.sync()
    r_loc = b_np - dy.numpy()
    sums = torch.tensor([float(r_loc @ r_loc), float(b_np @ b_np)], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(sums)
    true_res = float(torch.sqrt(sums[0] / sums[1]))
    ok = reason > 0 and true_res <= 1.01 * RTOL          # the TRUE residual, not the recurrence's estimate
    if args.dump_outputs:
        # each rank writes its own rows of x; the residual history is the same on every rank
        outputs = {"x" if world == 1 else "x_rank%d" % rank: xs}
        if rank == 0:
            outputs["residual_history"] = history
        dump_outputs(args.dump_outputs, outputs, DUMP_BYTES // world)

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        return
    peak, peak_src = peaks()
    achieved = (op_bytes / 1e9) / (op_ms / 1e3 / max(op_calls, 1)) if op_calls else None
    # dominant kernel: the Chebyshev-step launch of the BSR kernel on P_ss (level 0 of the solid V-cycle) -- the launch with
    # the largest share of a solve (ncu launch list in profiles/).  It is timed live by CUDA events on the library's stream
    # around every such launch of the profiled solves (slot 37); bytes = one product with P_ss in its launched format plus
    # the epilogue's vector traffic (r, d, D^-1, x read; r, d, x written: 56 B per row).
    parts = ksp.parts_info()
    FORMATS = {0: "CSR", 1: "BSR3", 2: "diag-BSR3", 3: "fused BSR3 + mass coupling"}
    dom = None
    try:
        ss_bytes, ss_fmt = pc.getPythonContext().block_bytes("ss")
        ns_rows = pc.getPythonContext().block_info("ss")[0]
        if 37 in phases and phases[37][1] > 0:
            ms37, n37 = phases[37]
            nbytes = ss_bytes + 56 * ns_rows
            dom = {"bytes": nbytes, "format": FORMATS.get(ss_fmt, "?"), "avg_ms": ms37 / n37, "launches": n37,
                   "achieved": nbytes / 1e9 / (ms37 / n37 / 1e3)}
    except Exception as e:
        print("[bench] dominant-kernel profile unavailable: %r" % (e,), file=sys.stderr)
    stats = pc.getPythonContext().stats()
    # value: device time (CUDA events); e2e: host wall clock around the K host-buffer calls (what a caller observes)
    t_solve, t_solve_e = dt / args.steps, max(dt_e, wall["e2e"]) / args.steps
    line = {
        "metric": METRIC, "value": n_global / t_solve if ok else None, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_solve, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(N, n_global, nnzA, maxiter, "maxiter", world),
                   "l2": "inputs larger than L2 (matrix streams >> 126 MB); no explicit flush",
                   "parallelism": "z-slab row partition x%d, distributed SA-AMG hierarchies" % world if world > 1 else "single GPU"},
        "wall_ms_per_step": 1e3 * wall["dev"] / args.steps, "time_to_1e-8_s": t_solve, "its_per_solve": its / args.steps, "its_per_s": its / dt,
        "dof_its_per_s": n_global * its / dt,
        "reason": reason, "rnorm": rnorm, "true_rel_residual": true_res, "converged": bool(ok),
        "setup_s": {"system_generation": t_asm, "generated_on": args.assemble, "pc_and_solver_setup": t_set},
        "inner": {k: v for k, v in stats.items() if k.startswith("its_") or k.startswith("calls_")},
        "e2e": {"value": n_global / t_solve_e if ok else None, "unit": UNIT, "h2d_bytes_per_step": int(b_host.numel() * 8),
                "d2h_bytes_per_step": int(x_host.numel() * 8), "ms_per_step": 1e3 * t_solve_e},
        "gpu_launches": int(launches),
        "profiled_pass": {"steps": prof_steps, "ms_per_step": 1e3 * dt_p / prof_steps,
                          "note": "separate pass with CUDA events on; phases, outer_operator and roofline come from it"},
        "phases_ms_per_solve": {PHASE_NAMES.get(k, str(k)): round(v[0] / prof_steps, 3) for k, v in sorted(phases.items())},
        "clocks": clocks,
    }
    if extra:
        line["config"]["extra_options"] = extra
    if dom:
        traffic, traffic_src = measured_traffic("s_L0_cheby_step", dom["bytes"])
        line["roofline"] = {"bound": "hbm", "kernel": "k_bsr_stream<3, mode 3 (Chebyshev step), PREF> on P_ss (%s), level 0 of the solid V-cycle: "
                                                      "the launch with the largest share of the solve" % dom["format"],
                            "achieved": dom["achieved"], "peak": peak, "unit": "GB/s", "frac": dom["achieved"] / peak,
                            "traffic": traffic, "traffic_source": traffic_src,
                            "peak_source": peak_src, "bytes_per_launch": dom["bytes"], "format": dom["format"],
                            "launches_timed": dom["launches"], "avg_launch_ms": dom["avg_ms"],
                            "frac_of_nominal_8TBs": dom["achieved"] / 8000.0}
    else:
        line["roofline"] = {"bound": "hbm", "kernel": "outer operator y = A x", "achieved": achieved, "peak": peak, "unit": "GB/s",
                            "frac": (achieved / peak) if achieved else None, "traffic": None, "peak_source": peak_src,
                            "bytes_per_launch": op_bytes, "launches_timed": op_calls, "avg_launch_ms": op_ms / max(op_calls, 1)}
    line["outer_operator"] = {"launches_per_product": len(parts), "bytes_per_product": op_bytes, "avg_ms": op_ms / max(op_calls, 1),
                              "achieved_GBs": achieved, "frac": (achieved / peak) if achieved else None,
                              "frac_of_nominal_8TBs": (achieved / 8000.0) if achieved else None,
                              "parts": [{"bytes": b, "format": FORMATS.get(f, "?")} for b, f in parts]}
    if not args.no_cpu_baseline and world == 1 and N <= args.cpu_max_n:
        try:
            line["cpu_baseline"] = cpu_baseline(N, xs)
            line["its_gpu_vs_cpu"] = [its / args.steps, line["cpu_baseline"]["its"]]
        except Exception as e:                  # never lose the measured GPU line over the CPU leg
            print("[bench] cpu_baseline failed: %r" % (e,), file=sys.stderr)
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    if not ok:
        print("[bench] solve did not converge: reason %d, true residual %.3e" % (reason, true_res), file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
