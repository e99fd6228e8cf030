#!/usr/bin/env python
"""bench.py -- headline benchmark of the ParMGMC sampling hot path on B200.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU arithmetic (oracle port) on the host cores

Workload (BASELINE.json configs[1]): 2D 5-point 4097x4097 shifted-Laplacian GMRF (src/problems.c:14-75 semantics),
PCGAMGMC V(1,1) cycle with SOR-Gibbs smoothers, Galerkin geometric hierarchy, dense Cholesky sampler on the coarsest level;
b = 0 (prior sampling, examples/ex8.c:47-49), device Philox noise.  One "step" = `--samples-per-step` MGMC samples (outer
Richardson iterations, src/pc_gamgmc.c:242-259) in ONE call of the sampler (KSPSolve with -ksp_max_it S).  For N > 1 the
grid is weak-scaled in y (one 4097 x 4096 slab per rank, halo exchange over NCCL); a unit of work is one sample of one
4097^2-DOF slab, so `value` = N * samples/s of the N-slab grid; the reference arm samples the SAME N-slab grid on the CPU.

One JSON line.  Beyond the contract's keys:
  roofline          the kernel with the largest share of the timed sample (per-kernel CUDA-event profile of the same sampler,
                    pmg_pc_profile), against the COMPULSORY bytes of that fused kernel (what a perfect implementation of the same
                    fusion must move: never above 1); `survey_bytes_frac` uses the sum of SURVEY 8(d)'s per-unit figures of the
                    passes the kernel replaces (K1 = 24 B at omega = 1), which fusion can exceed
  roofline_vcycle   the whole sample: sum over launches of the byte table / ms_per_sample / peak (table in DESIGN.md section 3)
  kernels           the profile itself (share, GB/s per kernel)
  multi_chain       N = 1: throughput of 4 independent chains of the headline sampler sharing the GPU (informational; `value` is ONE chain)
  gibbs2d, gibbs3d  stand-alone fused red-black sweeps (K1, 24 B / DOF-update at omega = 1), 4097^2 and 512^3 per GPU
  csr_sweep         K2: assembled 7-point 256^3 operator, SELL colour sweep (N = 1)
  mgmc3d            config 4's V-cycle: 513 x 513 x (512 N + 1), z-slabs
  parity_check      (N > 1) small slab / row-partitioned cases gathered on rank 0: bitwise against one GPU, 1e-12 against the oracle
  cpu_baseline      (N = 1, rank 0) the oracle port on the host: (i) 1 thread, the reference's 1-rank V-cycle; (ii) T threads
                    emulating T ranks of MCSORApply_MPIAIJ (row blocks + per-colour ghost exchange)
The oracle is used only as checker / CPU baseline (parity_check, cpu_baseline, --impl reference).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def grid_of(args, nranks):
    n = args.n
    return (n, n) if nranks == 1 else (n, (n - 1) * nranks + 1)


def workload_config(args, nranks):
    """The same dictionary for both arms (what differs between them is under `impl_notes`, outside `config`)."""
    n = args.n
    g = grid_of(args, nranks)
    return {"workload": f"2D 5-point {n}x{n} shifted-Laplacian GMRF per GPU, PCGAMGMC V(1,1), SOR-Gibbs smoother, Galerkin Q1 hierarchy, dense Cholesky coarsest",
            "grid_per_gpu": [n, n if nranks == 1 else n - 1], "grid_global": list(g), "kappa": args.kappa, "levels": args.levels,
            "rhs": "b = 0 (prior sampling)",
            "l2": "working set (>= 134 MB per fine vector, > 1 GB per sample) exceeds the 126 MB L2; no explicit flush",
            "parallelism": f"row-slab x{nranks}" if nranks > 1 else "single GPU"}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (oracle port: the checker's arithmetic, timed as the reference's CPU path)
# ---------------------------------------------------------------------------------------------------------------------
def cpu_baseline_leg(args, samples):
    """(i) the reference's 1-rank V-cycle on one thread; (ii) T threads emulating T ranks of MCSORApply_MPIAIJ."""
    import oracle as orc
    n = args.n
    t0 = time.time()
    mg = orc.MG.geometric(2, n, n, 1, args.kappa, args.levels)
    mg.setup()
    setup_s = time.time() - t0
    b, y = np.zeros(n * n), np.zeros(n * n)
    ns = orc.Noise.rander48()
    mg.richardson(ns, b, y, 1)  # warm caches / page in
    t0 = time.time()
    mg.richardson(ns, b, y, samples)
    dt = time.time() - t0
    out = {"value": samples / dt, "unit": "samples/s", "cores": 1, "kind": "port",
           "sample": f"{samples} MGMC samples of the full {n}x{n} workload after 1 warm-up sample (setup {setup_s:.1f} s not timed); "
                     "single thread = the reference's 1-rank path (one-colour lexicographic sweeps, rander48 Box-Muller)",
           "ms_per_sample": 1e3 * dt / samples}
    del mg
    # (ii) SURVEY 8(d)(ii): T threads = T ranks of MCSORApply_MPIAIJ (src/mc_sor.c:298-381): row blocks, red-black colouring,
    # per-colour ghost gather through shared memory; deterministic sweeps of the same 4097^2 operator (K2 bytes: 108 B / row)
    try:
        T = max(1, min(os.cpu_count() or 1, args.cpu_threads if args.cpu_threads > 0 else 64))
        A = orc.laplace(2, n, n, 1, args.kappa)
        col = orc.Coloring.parity((n, n))
        starts = np.round(np.linspace(0, A.n, T + 1)).astype(np.int64)
        part = orc.Partitioned(A, starts, col, 1.0)
        bb, yy = np.zeros(A.n), np.zeros(A.n)
        part.sweep(bb, yy, orc.SOR_FORWARD, nthreads=T)
        reps = 0
        t0 = time.time()
        while reps < 40 and time.time() - t0 < 8.0:
            part.sweep(bb, yy, orc.SOR_FORWARD, nthreads=T)
            reps += 1
        dts = (time.time() - t0) / reps
        out["mpiaij_sweep"] = {"value": A.n / dts, "unit": "DOF-updates/s", "cores": T, "kind": "port", "ms_per_sweep": 1e3 * dts,
                               "K2_GBs": 108.0 * A.n / dts / 1e9,
                               "sample": f"{reps} forward red-black sweeps of the {n}x{n} CSR operator, {T} threads emulating {T} ranks of MCSORApply_MPIAIJ (row blocks, per-colour ghost gather), no noise"}
    except Exception as e:  # the baseline must never take the bench line down
        out["mpiaij_sweep"] = {"error": repr(e)}
    return out


def _ref_worker(nx, ny, kappa, levels, per_step, warmup, steps, budget_s, start_evt, ready_q, done_q):
    """One independent chain of the reference's 1-rank CPU arithmetic (what a rank of `mpirun -np T` replicas would run)."""
    import oracle as orc
    mg = orc.MG.geometric(2, nx, ny, 1, kappa, levels)
    mg.setup()
    b, y = np.zeros(nx * ny), np.zeros(nx * ny)
    ns = orc.Noise.rander48()
    for _ in range(warmup):
        mg.richardson(ns, b, y, per_step)
    ready_q.put(1)
    start_evt.wait()
    t0 = time.time()
    done = 0
    for _ in range(steps):
        mg.richardson(ns, b, y, per_step)
        done += 1
        if time.time() - t0 > budget_s:  # bounded sample: stop early rather than run for tens of minutes on large N
            break
    done_q.put((time.time() - t0, done))


def run_reference(args):
    """The reference's CPU path on the box's host cores, on the b200 arm's configuration (the same global grid and level
    count at every N).  PETSc + MPI cannot be built here (DESIGN.md section 6), so the arithmetic is the oracle port of the
    1-rank reference; to use every host thread it runs T independent chains (the replica-parallel pattern of
    examples/ex7.c:136-205), T = min(cores, --ref-procs, memory / chain footprint)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    N = max(1, args.gpus)
    nx, ny = grid_of(args, N)
    per_step = max(1, args.ref_samples_per_step)
    cores = os.cpu_count() or 1
    try:
        mem_gb = os.sysconf("SC_PHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2 ** 30
    except (ValueError, OSError):
        mem_gb = 16.0
    per_proc_gb = 3.0 * (nx * ny) / 4097.0 ** 2
    T = max(1, min(cores, args.ref_procs if args.ref_procs > 0 else 16, int(mem_gb * 0.6 / per_proc_gb)))
    warm = 1 if N > 1 else min(args.warmup, 3)
    mpc = mp.get_context("spawn")
    start_evt, ready_q, done_q = mpc.Event(), mpc.Queue(), mpc.Queue()
    procs = [mpc.Process(target=_ref_worker, args=(nx, ny, args.kappa, args.levels, per_step, warm, args.steps, args.ref_budget_s, start_evt, ready_q, done_q)) for _ in range(T)]
    for p in procs:
        p.start()
    for _ in range(T):
        ready_q.get()
    start_evt.set()
    res = [done_q.get() for _ in range(T)]
    for p in procs:
        p.join()
    # every chain reports (its own time, steps done); units of work: one sample of one 4097^2 slab = N units per sample
    value = sum(N * d * per_step / t for t, d in res)
    steps_done = min(d for _, d in res)
    slowest = max(t for t, _ in res)
    cfg = workload_config(args, N)
    out = {"impl": "reference", "metric": "mgmc_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": args.gpus, "steps": steps_done, "steps_requested": args.steps,
           "warmup": warm, "ms_per_step": 1e3 * slowest / max(1, steps_done), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": cfg, "samples_per_step": per_step,
           "impl_notes": {"parallelism": f"{T} independent CPU chains (one per host thread used), each sampling the whole {nx}x{ny} grid",
                          "noise": "rander48 Box-Muller (PETSc's default PetscRandom, src/parmgmc.c:100-110)",
                          "sweep_order": "lexicographic, the reference's 1-rank order (src/mc_sor.c:397-410)",
                          "unit_of_work": "one sample of one 4097^2-DOF slab (a sample of the N-slab grid counts N)"},
           "cpu_baseline": {"value": value, "unit": "samples/s", "cores": T, "kind": "port", "host_cores": cores,
                            "sample": f"{T} chains x {steps_done} step(s) x {per_step} sample(s) of the full {nx}x{ny} workload (slowest chain {slowest:.1f} s, per-chain budget {args.ref_budget_s:.0f} s); "
                                      "the reference (PETSc+MPI) cannot be built here, so each chain is the oracle port of its 1-rank path"},
           "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(out)


# ---------------------------------------------------------------------------------------------------------------------
# multi-GPU parity check (runs before the timed region at N > 1)
# ---------------------------------------------------------------------------------------------------------------------
def parity_check(pmg, ctx, rank, world, local):
    """Slab-partitioned samplers over NCCL, gathered on rank 0 and compared BITWISE with one GPU (Philox is keyed on the
    global index, so the result may not depend on the partition), plus the one-GPU path against the CPU oracle (1e-12), plus a
    row-partitioned CSR operator (MCSORApply_MPIAIJ) against the oracle's emulation of it."""
    import torch.distributed as dist
    cases = []
    ok_all = True

    def slab_case(name, pctype, dim, dims, opts, its):
        nonlocal ok_all
        nslow = dims[2] if dim == 3 else dims[1]
        slab = pmg.partition_slabs(nslow, world)[rank]
        n = dims[0] * dims[1] * dims[2]
        rng = np.random.default_rng(99)
        b_full, y0 = rng.standard_normal(n), rng.standard_normal(n)

        def run(c, sl):
            mat = pmg.Mat.laplace(c, dim, dims[0], dims[1], dims[2], kappa=1.0, slab=sl)
            nloc, _, row0 = mat.size
            pc = pmg.PC(c, pctype)
            pc.set_operator(mat)
            pc.set_options(dict(opts, **{"-pc_b200_noise": "philox"}))
            pc.setup()
            c.set_seed(4242)
            y = y0[row0:row0 + nloc].copy()
            pc.apply_richardson(b_full[row0:row0 + nloc].copy(), y, its=its)
            return row0, y

        row0, y = run(ctx, slab)
        parts = [None] * world
        dist.all_gather_object(parts, (row0, y))
        rec = None
        if rank == 0:
            import oracle as orc
            got = np.empty(n)
            for r0, yy in parts:
                got[r0:r0 + yy.size] = yy
            single = pmg.Context(local, seed=4242)
            _, ref = run(single, None)
            bitwise = bool(np.array_equal(got, ref))
            # the one-GPU path against the oracle
            if pctype == "gamgmc":  # injected tape (the oracle's V-cycle takes the reference's tape order, SURVEY 8(c))
                L = int(opts["-gamgmc_pc_mg_levels"])
                pc = pmg.PC(single, "gamgmc")
                pc.set_operator(pmg.Mat.laplace(single, dim, *dims, kappa=1.0))
                pc.set_options(dict(opts))
                pc.setup()
                z = rng.standard_normal(its * pc.noise_per_sample())
                pc.set_noise_tape(z)
                yt = y0.copy()
                pc.apply_richardson(b_full, yt, its=its)
                omg = orc.MG.geometric(dim, dims[0], dims[1], dims[2], 1.0, L)
                for l in range(1, L):
                    d = omg.level_dims(l)
                    omg.set_smoother(l, orc.KIND_SORGIBBS, 1.0, orc.SOR_FORWARD, 1, orc.Coloring.parity(d[:dim], 2 if l == L - 1 else 2 ** dim))
                omg.setup()
                oref = omg.richardson(orc.Noise.tape(z), b_full, y0.copy(), its)
                oerr = float(np.abs(yt - oref).max() / np.abs(oref).max())
            else:  # device Philox against the oracle's Philox definition
                A = orc.laplace(dim, *dims, kappa=1.0)
                col = orc.Coloring.parity(dims[:dim])
                sweep = orc.SOR_SYMMETRIC if "-pc_mcgibbs_symmetric" in opts else orc.SOR_FORWARD
                oref = orc.gibbs_richardson(A, b_full, y0.copy(), its, orc.Noise.philox(4242, dims), col, float(opts.get("-pc_mcgibbs_omega", 1.0)), sweep)
                oerr = float(np.abs(ref - oref).max() / np.abs(oref).max())
            ok = bitwise and oerr < 1e-12
            rec = {"case": name, "bitwise_vs_one_gpu": bitwise, "one_gpu_vs_oracle_relerr": oerr, "ok": bool(ok)}
            single.close()
        return rec

    def csr_case():
        import oracle as orc
        import scipy.sparse as sp
        A0 = orc.laplace(2, 33, 29, kappa=1.0)
        n = A0.n
        rng = np.random.default_rng(7)
        perm = rng.permutation(n)
        M = sp.csr_matrix(A0.to_scipy())[perm][:, perm].tocsr()
        M.sort_indices()
        A = orc.CSR(n, M.indptr.astype(np.int64), M.indices.astype(np.int32), M.data.astype(np.float64))
        starts = np.round(np.linspace(0, n, world + 1)).astype(np.int64)
        r0, r1 = int(starts[rank]), int(starts[rank + 1])
        rp = (M.indptr[r0:r1 + 1] - M.indptr[r0]).astype(np.int64)
        mat = pmg.Mat.from_csr_dist(ctx, n, r0, rp, M.indices[M.indptr[r0]:M.indptr[r1]].astype(np.int64), M.data[M.indptr[r0]:M.indptr[r1]].astype(np.float64))
        gcol = orc.Coloring.greedy(A)
        mat.set_coloring(gcol.color[r0:r1], gcol.ncolors)
        b_full, y0 = rng.standard_normal(n), rng.standard_normal(n)
        mc = pmg.MCSOR(mat)
        mc.set_omega(1.3)
        mc.set_sweep_type(3)
        ys = y0[r0:r1].copy()
        mc.apply(b_full[r0:r1].copy(), ys)
        parts = [None] * world
        dist.all_gather_object(parts, (r0, ys))
        if rank != 0:
            return None
        got = np.empty(n)
        for q0, yy in parts:
            got[q0:q0 + yy.size] = yy
        ref = y0.copy()
        orc.Partitioned(A, starts, gcol, 1.3).sweep(b_full, ref, orc.SOR_SYMMETRIC, nthreads=world)
        err = float(np.abs(got - ref).max())
        return {"case": f"csr_dist 957 rows on {world} ranks, MCSORApply symmetric omega 1.3 vs oracle MCSORApply_MPIAIJ", "abs_err": err, "ok": bool(err < 1e-12)}

    for rec in (slab_case("gibbs3d 33x24x40 mcgibbs symmetric omega 1.3", "mcgibbs", 3, (33, 24, 40), {"-pc_mcgibbs_symmetric": "", "-pc_mcgibbs_omega": 1.3}, 2),
                slab_case("gamgmc2d 129x257 4 levels", "gamgmc", 2, (129, 257, 1), {"-gamgmc_pc_mg_levels": 4}, 2),
                slab_case("gamgmc3d 33x33x65 3 levels", "gamgmc", 3, (33, 33, 65), {"-gamgmc_pc_mg_levels": 3}, 2),
                csr_case()):
        if rank == 0:
            cases.append(rec)
            ok_all = ok_all and rec["ok"]
    return {"cases": cases, "ok": bool(ok_all)} if rank == 0 else None


def assemble_laplace3d_csr(n, kappa):
    """7-point shifted Laplacian of src/problems.c:14-75 extended to 3D (SURVEY F8), assembled with numpy (no oracle here)."""
    idx = np.arange(n ** 3, dtype=np.int64)
    i, j, k = idx % n, (idx // n) % n, idx // (n * n)
    h = 1.0 / (n - 1) ** 2
    offs = [(-n * n, k > 0), (-n, j > 0), (-1, i > 0), (0, None), (1, i < n - 1), (n, j < n - 1), (n * n, k < n - 1)]
    deg = sum(m.astype(np.int64) for _, m in offs if m is not None)
    cols = np.empty((n ** 3, 7), dtype=np.int32)
    vals = np.empty((n ** 3, 7), dtype=np.float64)
    mask = np.empty((n ** 3, 7), dtype=bool)
    for q, (o, m) in enumerate(offs):
        cols[:, q] = (idx + o).astype(np.int32)
        if m is None:
            d = np.full(n ** 3, kappa * kappa)
            for t in range(1, 7):
                d = np.where(deg >= t, d + h, d)  # one += per existing neighbour (src/problems.c:31-58)
            vals[:, q], mask[:, q] = d, True
        else:
            vals[:, q], mask[:, q] = -h, m
    rowptr = np.zeros(n ** 3 + 1, dtype=np.int64)
    np.cumsum(mask.sum(axis=1), out=rowptr[1:])
    return rowptr, cols[mask], vals[mask], ((i + j + k) & 1).astype(np.int32)


DUMP_ENTRIES = 1 << 22  # 32 MiB of float64 over all ranks


def dump_outputs(path, y, rank, world):
    """Writes the chain state y after the last timed step -- what apply_richardson_dev hands back to its caller -- as
    <path>/y.npy (float64; y_rank<r>.npy per rank for N > 1).  A state longer than its share of DUMP_ENTRIES is written as the
    entries at a fixed sorted sample of indices (seed 0, so the same indices for the same grid), so that the dumps of two builds
    can be compared entry for entry."""
    os.makedirs(path, exist_ok=True)
    v = y.cpu().numpy()
    cap = DUMP_ENTRIES // world
    if v.size > cap:
        v = v[np.sort(np.random.default_rng(0).choice(v.size, cap, replace=False))]
    np.save(os.path.join(path, "y.npy" if world == 1 else f"y_rank{rank}.npy"), v)


def run_b200(args):
    import torch
    import torch.distributed as dist

    import parmgmc_b200 as pmg

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.current_stream()
    ctx = pmg.Context(local, stream=stream.cuda_stream, seed=0xCAFE)
    if world > 1:
        uid = [pmg.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- multi-GPU correctness first: a number from a wrong distributed path is worth nothing ----
    parity = None
    if world > 1 and not args.no_parity_check:
        def _checked():
            p = parity_check(pmg, ctx, rank, world, local)
            f = torch.tensor([0 if (p is None or p["ok"]) else 1], device="cuda")
            dist.broadcast(f, src=0)
            return p, int(f.item())
        parity, bad = _checked()
        if bad and "PMG_NO_OVERLAP_SWEEP" not in os.environ:
            # the newest distributed path (boundary bands of the 2D sweeps on the communication stream) has a switch: measure without it
            # rather than not at all, and say so in the line
            first = parity
            os.environ["PMG_NO_OVERLAP_SWEEP"] = "1"
            parity, bad = _checked()
            if rank == 0 and parity is not None:
                parity["fallback"] = {"PMG_NO_OVERLAP_SWEEP": "1", "failed_with_overlap": first}
        if bad:
            if rank == 0:
                _emit({"metric": "mgmc_samples_per_s", "error": "multi-GPU parity check failed", "parity_check": parity})
            dist.destroy_process_group()
            sys.exit(1)
        ctx.set_seed(0xCAFE)

    n = args.n
    nx, ny = grid_of(args, world)
    slab = pmg.partition_slabs(ny, world)[rank] if world > 1 else None
    mat = pmg.Mat.laplace(ctx, 2, nx, ny, 1, args.kappa, slab=slab)
    pc = pmg.PC(ctx, "gamgmc")
    pc.set_operator(mat)
    pc.set_options({"-gamgmc_pc_mg_levels": args.levels, "-pc_b200_noise": "philox"})
    t0 = time.time()
    pc.setup()
    setup_s = time.time() - t0
    nloc = mat.n
    S = args.samples_per_step
    peak, peak_src = measured_peaks()

    y = torch.zeros(nloc, dtype=torch.float64, device="cuda")
    b = torch.zeros(nloc, dtype=torch.float64, device="cuda")

    # ---- device-resident throughput ("value") ----
    for _ in range(args.warmup):
        pc.apply_richardson_dev(b, y, its=S)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = updates = 0
    e0.record(stream)
    for _ in range(args.steps):
        pc.apply_richardson_dev(b, y, its=S)
        st = pc.last_stats()
        launches += st["launches"]; updates += st["dof_updates"]
    e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    value = world * args.steps * S / (ms * 1e-3)
    ms_per_sample = ms / (args.steps * S)
    if args.dump_outputs:  # before the legs below, which advance the same chain state
        dump_outputs(args.dump_outputs, y, rank, world)

    # ---- end to end through the host-pointer C-ABI call: pinned host buffers, H2D of the chain state y (b = NULL: the zero
    #      right-hand side of prior sampling is never uploaded), S samples, D2H of y, all inside the timed region ----
    hy = torch.zeros(nloc, dtype=torch.float64).pin_memory().numpy()
    pc.apply_richardson(None, hy, its=S)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    e0.record(stream)
    for _ in range(e2e_steps):
        pc.apply_richardson(None, hy, its=S)
    e1.record(stream)
    barrier()
    e2e_value = world * e2e_steps * S / (max_over_ranks(e0.elapsed_time(e1)) * 1e-3)

    # ---- per-kernel profile of the same sampler (CUDA events around every launch of the V-cycle, same stream) ----
    kernels, roofline, roofline_vcycle = [], None, None
    try:
        pc.set_option("-pc_b200_profile", 1)
        pc.apply_richardson_dev(b, y, its=4)
        pc.profile(reset=True)
        nprof = 20
        pc.apply_richardson_dev(b, y, its=nprof)
        prof = pc.profile(reset=True)
        pc.set_option("-pc_b200_profile", 0)
        tot_ms = sum(k["ms"] for k in prof) or 1.0
        for k in prof:
            per_launch_ms = k["ms"] / max(1, k["launches"])
            kernels.append({"kernel": k["kernel"], "launches_per_sample": k["launches"] / nprof, "us_per_launch": 1e3 * per_launch_ms, "share": k["ms"] / tot_ms,
                            "compulsory_GBs": (k["bytes_min"] / max(1, k["launches"])) / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else None,
                            "survey_GBs": (k["bytes_survey"] / max(1, k["launches"])) / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else None})
        dom = max(kernels, key=lambda k: k["share"]) if kernels else None
        if dom is not None and dom["compulsory_GBs"]:
            traffic, traffic_src = None, None
            tj = os.path.join(ROOT, "profiles", "r2_traffic.json")
            if world == 1 and os.path.exists(tj):
                t = json.load(open(tj))
                ent = t.get("kernels", {}).get(dom["kernel"])
                if ent and t.get("n") == n:
                    traffic, traffic_src = ent.get("dram_bytes_per_launch"), t.get("source")
            roofline = {"bound": "hbm", "achieved": dom["compulsory_GBs"], "peak": peak, "unit": "GB/s", "frac": dom["compulsory_GBs"] / peak, "traffic": traffic, "traffic_source": traffic_src,
                        "kernel": dom["kernel"], "share_of_sample": dom["share"], "launch_ms": dom["us_per_launch"] * 1e-3,
                        "bytes_model": "compulsory bytes of the fused kernel (b in, x in unless zero, x out, coarse vector in / out): what a perfect implementation of this fusion moves",
                        "survey_bytes_GBs": dom["survey_GBs"], "survey_bytes_frac": dom["survey_GBs"] / peak,
                        "survey_bytes_model": "sum of SURVEY 8(d)'s per-unit figures of the passes the kernel replaces: K1 24 B (omega = 1) [+ K3 24 + K4 10 | + K5 18] per DOF",
                        "peak_source": peak_src, "frac_of_nominal_8TBs": dom["compulsory_GBs"] / 8000.0,
                        "timing": "CUDA events around each launch of this kernel inside the sampler, on the launching stream, averaged over 20 samples"}
            bmin = sum(k["bytes_min"] for k in prof) / nprof
            bsur = sum(k["bytes_survey"] for k in prof) / nprof
            roofline_vcycle = {"bound": "hbm", "unit": "GB/s", "peak": peak, "ms_per_sample": ms_per_sample,
                               "compulsory_bytes_per_sample": bmin, "achieved": bmin / (ms_per_sample * 1e-3) / 1e9, "frac": bmin / (ms_per_sample * 1e-3) / 1e9 / peak,
                               "survey_bytes_per_sample": bsur, "survey_bytes_GBs": bsur / (ms_per_sample * 1e-3) / 1e9, "survey_bytes_frac": bsur / (ms_per_sample * 1e-3) / 1e9 / peak,
                               "note": "bytes of the labelled launches (per-kernel table in DESIGN.md section 3) / the event-timed sample of the headline run; the coarse tail launch is counted with 0 bytes"}
    except Exception as e:  # an older library without the profile entry point must not take the line down
        kernels = [{"error": repr(e)}]
    view = pc.view().strip().splitlines()[:2]

    # ---- stand-alone fine-level colour sweep (K1, 2D): 24 B / DOF-update at omega = 1 (b in, x out, other colour's neighbours) ----
    gibbs = pmg.PC(ctx, "sorgibbs")
    gibbs.set_operator(mat)
    gibbs.set_option("-pc_b200_noise", "philox")
    gibbs.setup()
    for _ in range(3):
        gibbs.apply_richardson_dev(b, y, its=4)
    barrier()
    nsweeps = 40
    e0.record(stream)
    gibbs.apply_richardson_dev(b, y, its=nsweeps)
    e1.record(stream)
    barrier()
    sweep_ms = max_over_ranks(e0.elapsed_time(e1)) / nsweeps
    bpu = args.bytes_per_update
    ach2 = bpu * nloc / (sweep_ms * 1e-3) / 1e9
    gibbs2d = {"workload": f"2D 5-point {nx}x{ny // world if world > 1 else ny} per GPU, fused red-black sweep (sweep2d_kernel), sorgibbs (omega = 1)", "sweep_ms": sweep_ms,
               "dof_updates_per_s": world * nloc / (sweep_ms * 1e-3),
               "roofline": {"bound": "hbm", "achieved": ach2, "peak": peak, "unit": "GB/s", "frac": ach2 / peak, "frac_of_nominal_8TBs": ach2 / 8000.0, "algorithmic_bytes_per_dof_update": bpu}}
    del gibbs, pc

    # ---- BASELINE's target kernel: the fused 3D 7-point sweep on 512^3 per GPU (z-slabs, NCCL halo for N > 1) ----
    gibbs3d = None
    if not args.no_gibbs3d:
        n3 = args.n3
        nz = n3 * world
        slab3 = pmg.partition_slabs(nz, world)[rank] if world > 1 else None
        mat3 = pmg.Mat.laplace(ctx, 3, n3, n3, nz, args.kappa, slab=slab3)
        g3 = pmg.PC(ctx, "sorgibbs")
        g3.set_operator(mat3)
        g3.set_option("-pc_b200_noise", "philox")
        g3.setup()
        y3 = torch.zeros(mat3.n, dtype=torch.float64, device="cuda")
        b3 = torch.zeros(mat3.n, dtype=torch.float64, device="cuda")
        g3.apply_richardson_dev(b3, y3, its=3)
        barrier()
        e0.record(stream)
        g3.apply_richardson_dev(b3, y3, its=20)
        e1.record(stream)
        barrier()
        ms3 = max_over_ranks(e0.elapsed_time(e1) / 20)
        ach3 = bpu * mat3.n / (ms3 * 1e-3) / 1e9
        gibbs3d = {"workload": f"3D 7-point {n3}^3 per GPU, fused red-black sweep with a right-hand side (sweep3d_kernel, warp-specialised, one CTA per tile), sorgibbs (omega = 1)", "sweep_ms": ms3, "dof_updates_per_s": world * mat3.n / (ms3 * 1e-3),
                   "roofline": {"bound": "hbm", "achieved": ach3, "peak": peak, "unit": "GB/s", "frac": ach3 / peak, "frac_of_nominal_8TBs": ach3 / 8000.0, "algorithmic_bytes_per_dof_update": bpu}}
        # prior sampling (b = NULL: nothing to read but the iterate): the persistent warp-specialised kernel (sweep3d_ws.cuh), 16 B / update
        if world == 1:
            g3.apply_richardson_dev(None, y3, its=3)
            e0.record(stream)
            g3.apply_richardson_dev(None, y3, its=20)
            e1.record(stream)
            torch.cuda.synchronize()
            ms3n = e0.elapsed_time(e1) / 20
            ach3n = 16.0 * mat3.n / (ms3n * 1e-3) / 1e9
            gibbs3d["no_rhs"] = {"workload": "the same sweep with b = NULL (prior sampling; sweep3d_ws_kernel, persistent)", "sweep_ms": ms3n, "dof_updates_per_s": mat3.n / (ms3n * 1e-3),
                                 "roofline": {"bound": "hbm", "achieved": ach3n, "peak": peak, "unit": "GB/s", "frac": ach3n / peak, "algorithmic_bytes_per_dof_update": 16.0}}
        del g3, mat3, y3, b3

    # ---- config 4: MGMC V-cycle on a 3D grid, 513 x 513 x (512 N + 1), z-slabs, dense Cholesky coarsest ----
    mgmc3d = None
    if not args.no_mgmc3d:
        try:
            nm = args.n3 + 1 if args.n3 % 2 == 0 else args.n3  # 2^k + 1 nodes per direction for the Q1 hierarchy
            nzm = (nm - 1) * world + 1
            lv3 = 1
            d = [nm, nm, nzm]
            while all((q - 1) % 2 == 0 for q in d) and d[0] * d[1] * d[2] > 4096:
                d = [(q + 1) // 2 for q in d]
                lv3 += 1
            slabm = pmg.partition_slabs(nzm, world)[rank] if world > 1 else None
            matm = pmg.Mat.laplace(ctx, 3, nm, nm, nzm, args.kappa, slab=slabm)
            m3 = pmg.PC(ctx, "gamgmc")
            m3.set_operator(matm)
            m3.set_options({"-gamgmc_pc_mg_levels": lv3, "-pc_b200_noise": "philox"})
            m3.setup()
            ym = torch.zeros(matm.n, dtype=torch.float64, device="cuda")
            bm = torch.zeros(matm.n, dtype=torch.float64, device="cuda")
            m3.apply_richardson_dev(bm, ym, its=2)
            barrier()
            e0.record(stream)
            its3 = 16  # one call: the layout copies of b and y (odd row length -> pitched copies) are paid once per call
            m3.apply_richardson_dev(bm, ym, its=its3)
            e1.record(stream)
            barrier()
            msm = max_over_ranks(e0.elapsed_time(e1)) / its3
            # bytes per sample and fine DOF: SURVEY 8(d)'s literal form at omega = 1 (K3 24 + 2 K1 24 + K3 24 + K4 9 + K5 17 + 2 K6 24 = 170) and
            # the compulsory traffic of the passes this implementation runs (2 sweeps 24 + residual 24 + restriction 9 + prolongation 17 = 98),
            # both times the level series 8/7
            ndof = float(matm.n)
            sv, cp = 170.0 * ndof * 8.0 / 7.0, 98.0 * ndof * 8.0 / 7.0
            mgmc3d = {"workload": f"3D 7-point {nm}x{nm}x{nzm} ({nm}x{nm}x{nm - 1 if world > 1 else nm} per GPU), PCGAMGMC V(1,1), {lv3} levels, SOR-Gibbs smoother, dense Cholesky coarsest ({d[0]}x{d[1]}x{d[2]})",
                      "ms_per_sample": msm, "samples_per_s": 1e3 / msm, "slab_samples_per_s": world * 1e3 / msm, "launches_per_sample": m3.last_stats()["launches"] / its3, "samples_per_call": its3,
                      "roofline": {"bound": "hbm", "peak": peak, "unit": "GB/s", "survey_bytes_per_sample": sv, "survey_GBs": sv / (msm * 1e-3) / 1e9, "survey_frac": sv / (msm * 1e-3) / 1e9 / peak,
                                   "compulsory_bytes_per_sample": cp, "compulsory_GBs": cp / (msm * 1e-3) / 1e9, "compulsory_frac": cp / (msm * 1e-3) / 1e9 / peak,
                                   "note": "per GPU; survey = SURVEY 8(d) literal per-pass byte counts, compulsory = what the passes of this implementation must move"}}
            del m3, matm, ym, bm
        except Exception as e:
            mgmc3d = {"error": repr(e)}

    # ---- independent chains on one GPU (what the reference arm does with its CPU cores): one stream, one context and one host
    # ---- thread per chain; the launch-latency-bound small levels of one chain run beside the other chains' kernels.  Reported
    # ---- beside the headline, which stays ONE chain ----
    multi_chain = None
    if world == 1 and not args.no_multi_chain:
        try:
            import threading
            chains = []
            for c in range(args.chains):
                st = torch.cuda.Stream()
                cx = pmg.Context(local, stream=st.cuda_stream, seed=0xCAFE + 1 + c)
                mt = pmg.Mat.laplace(cx, 2, nx, ny, 1, args.kappa)
                p2 = pmg.PC(cx, "gamgmc")
                p2.set_operator(mt)
                p2.set_options({"-gamgmc_pc_mg_levels": args.levels, "-pc_b200_noise": "philox"})
                p2.setup()
                yc = torch.zeros(mt.n, dtype=torch.float64, device="cuda")
                p2.apply_richardson_dev(None, yc, its=3)
                chains.append((st, cx, mt, p2, yc))
            torch.cuda.synchronize()
            ncall = 4

            def _work(ch):
                for _ in range(ncall):
                    ch[3].apply_richardson_dev(None, ch[4], its=S)

            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            th = [threading.Thread(target=_work, args=(ch,)) for ch in chains]
            for t in th:
                t.start()
            for t in th:
                t.join()
            torch.cuda.synchronize()
            eb.record()
            torch.cuda.synchronize()
            msc = ea.elapsed_time(eb)
            tot = args.chains * S * ncall
            multi_chain = {"workload": f"{args.chains} independent chains of the headline sampler on one GPU (one stream and one host thread each), {S} samples per call, {ncall} calls per chain",
                           "chains": args.chains, "samples": tot, "ms": msc, "samples_per_s": 1e3 * tot / msc, "ms_per_sample": msc / tot, "vs_one_chain": (1e3 * tot / msc) / value}
            del chains
        except Exception as e:
            multi_chain = {"error": repr(e)}

    # ---- K2: assembled-operator path, SELL colour sweep on the 7-point 256^3 operator (N = 1) ----
    csr_sweep = None
    if world == 1 and not args.no_csr:
        try:
            nc = args.n_csr
            rowptr, col, val, colour = assemble_laplace3d_csr(nc, args.kappa)
            matc = pmg.Mat.from_csr(ctx, rowptr, col, val)
            matc.set_coloring(colour, 2)
            nrows, nnz = nc ** 3, int(rowptr[-1])
            del rowptr, col, val, colour
            pcc = pmg.PC(ctx, "sorgibbs")
            pcc.set_operator(matc)
            pcc.set_option("-pc_b200_noise", "philox")
            pcc.setup()
            yc = torch.zeros(nrows, dtype=torch.float64, device="cuda")
            bc = torch.zeros(nrows, dtype=torch.float64, device="cuda")
            pcc.apply_richardson_dev(bc, yc, its=3)
            barrier()
            e0.record(stream)
            pcc.apply_richardson_dev(bc, yc, its=20)
            e1.record(stream)
            barrier()
            msc = e0.elapsed_time(e1) / 20
            brow = 12.0 * nnz / nrows + 48.0
            achc = brow * nrows / (msc * 1e-3) / 1e9
            csr_sweep = {"workload": f"3D 7-point {nc}^3 assembled CSR -> colour-sorted SELL, red-black, sorgibbs, Philox (sell_sweep_kernel, one launch per colour)", "sweep_ms": msc,
                         "dof_updates_per_s": nrows / (msc * 1e-3),
                         "roofline": {"bound": "hbm", "achieved": achc, "peak": peak, "unit": "GB/s", "frac": achc / peak, "algorithmic_bytes_per_row": brow, "model": "K2 of SURVEY 8(d): 12 nnz_row + 48 B / row"}}
            del pcc, matc, yc, bc
        except Exception as e:
            csr_sweep = {"error": repr(e)}

    if rank == 0:
        cpu = cpu_baseline_leg(args, args.cpu_samples) if (world == 1 and not args.no_cpu_baseline) else None
        out = {"metric": "mgmc_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": workload_config(args, world), "samples_per_step": S,
               "impl_notes": {"parallelism": (f"row-slab x{world}, ghost rows through peer memory over NVLink (CUDA IPC mailboxes, one kernel per exchange); NCCL for the gather of replicated levels"
                                               if ctx.comm_p2p() else f"row-slab x{world}, NCCL send/recv halo") if world > 1 else "single GPU", "noise": "device Philox4x32-10 + Box-Muller, keyed on the global index",
                              "sweep_order": "red-black on the fine level, four-colour on the Galerkin levels", "unit_of_work": "one sample of one 4097^2-DOF slab (a sample of the N-slab grid counts N)"},
               "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(8 * nloc), "d2h_bytes_per_step": int(8 * nloc),
                       "note": "per step: H2D of the chain state y from pinned memory, S samples, D2H of y; b = NULL (zero right-hand side, never uploaded)"},
               "gpu_launches": int(launches), "clocks": clk,
               "roofline": roofline, "roofline_vcycle": roofline_vcycle, "kernels": kernels,
               "setup_s": setup_s, "mgmc_ms_per_sample": ms_per_sample, "launches_per_sample": launches / (args.steps * S), "view": view,
               "gibbs2d": gibbs2d, "gibbs_dof_updates_per_s": gibbs2d["dof_updates_per_s"]}
        if gibbs3d is not None:
            out["gibbs3d"] = gibbs3d
        if mgmc3d is not None:
            out["mgmc3d"] = mgmc3d
        if csr_sweep is not None:
            out["csr_sweep"] = csr_sweep
        if multi_chain is not None:
            out["multi_chain"] = multi_chain
        if parity is not None:
            out["parity_check"] = parity
        if cpu is not None:
            out["cpu_baseline"] = cpu
        _emit(out)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def _protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout when the
    box sets NCCL_DEBUG=VERSION): everything but the JSON line goes to stderr."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def _emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=4097)
    ap.add_argument("--n3", type=int, default=512, help="edge of the 3D grid per GPU for the gibbs3d / mgmc3d measurements")
    ap.add_argument("--n-csr", type=int, default=256, help="edge of the assembled 3D operator of the K2 measurement")
    ap.add_argument("--levels", type=int, default=0, help="0: coarsen until the coarsest grid has at most --coarsest-max nodes (10 levels, 9x9, at N = 1)")
    ap.add_argument("--coarsest-max", type=int, default=100, help="largest coarsest grid of the automatic level count (dense Cholesky sampler there); 1200 gives round 1's 8 levels / 33x33")
    ap.add_argument("--kappa", type=float, default=1.0)
    ap.add_argument("--samples-per-step", type=int, default=120, help="MGMC samples per sampler call; 120 makes a step >= 50 ms")
    ap.add_argument("--ref-samples-per-step", type=int, default=1)
    ap.add_argument("--ref-procs", type=int, default=0, help="CPU chains of the reference arm (0: min(cores, 16, memory / chain footprint))")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="per-chain time budget of the reference arm's timed region")
    ap.add_argument("--no-gibbs3d", action="store_true", help="skip the 3D 7-point sweep measurement")
    ap.add_argument("--no-mgmc3d", action="store_true", help="skip the 3D V-cycle measurement")
    ap.add_argument("--no-csr", action="store_true", help="skip the assembled-operator (K2) measurement")
    ap.add_argument("--no-multi-chain", action="store_true", help="skip the concurrent-chains measurement (N = 1)")
    ap.add_argument("--chains", type=int, default=4, help="independent chains of the concurrent-chains measurement")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the multi-GPU parity check (N > 1)")
    ap.add_argument("--cpu-samples", type=int, default=4)
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the MPIAIJ-emulation CPU baseline (0: all host cores)")
    ap.add_argument("--bytes-per-update", type=float, default=24.0, help="algorithmic bytes per DOF update of the omega = 1 colour sweep (SURVEY 8(d) K1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the chain state after the last timed step to DIR/y.npy (a fixed sample of 2^22 entries when it is longer)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl b200)")
    if args.levels <= 0:  # coarsen until the coarsest grid is small (SURVEY 8(d): cut at <= 33x33 + dense Cholesky; 9x9 at N = 1: the levels up to 65x65 run in one shared-memory launch)
        nx, ny = grid_of(args, max(1, args.gpus))
        args.levels = 1
        while nx * ny > args.coarsest_max and (nx - 1) % 2 == 0 and (ny - 1) % 2 == 0 and min((nx + 1) // 2, (ny + 1) // 2) >= 3:
            nx, ny = (nx + 1) // 2, (ny + 1) // 2
            args.levels += 1
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
