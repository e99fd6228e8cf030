"""One rank of a multi-GPU run of low-rank-corrected (MATLRC) operators, launched by tests/test_multigpu_lrc.py with
torch.distributed.run, one process per GPU.  The base is distributed (a slab of a grid operator or the rows of a
row-partitioned CSR operator); B holds this rank's rows.  B^T y is a sum over all rows that is split at rank boundaries,
so N GPUs are compared with one GPU to rounding: max|dy| / max|y| <= 1e-12 with equal draw counters; a second run at the
same N must give the same bits."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import parmgmc_b200 as pmg  # noqa: E402

TOL = 1e-12

CASES = {
    # name: (pc type, dim, dims, options, its, ragged cut?, k)
    "mcgibbs2d_sym": ("mcgibbs", 2, (65, 67, 1), {"-pc_mcgibbs_symmetric": "", "-pc_mcgibbs_omega": 1.3}, 3, True, 5),
    "sorgibbs3d": ("sorgibbs", 3, (17, 12, 20), {}, 3, False, 4),
    "gamgmc2d": ("gamgmc", 2, (129, 257, 1), {"-gamgmc_pc_mg_levels": 4, "-pc_b200_replicate_below": 500}, 2, False, 6),
    "gamgmc3d": ("gamgmc", 3, (33, 33, 65), {"-gamgmc_pc_mg_levels": 3}, 2, False, 3),
}


def obs_matrix(rng, n, k):
    """k sparse positive observation columns (the _obs_matrix of test_gpu_parity.py)."""
    B = np.zeros((n, k))
    for j in range(k):
        idx = rng.choice(n, size=min(n, 12), replace=False)
        B[idx, j] = rng.uniform(0.2, 1.0, idx.size)
    return B


def slabs_for(dim, dims, world, ragged):
    nslow = dims[2] if dim == 3 else dims[1]
    slabs = pmg.partition_slabs(nslow, world, align=1 if ragged else 2)
    if ragged and world > 1:  # move the first cut to an odd unit
        lo, hi = slabs[0]
        slabs[0] = (lo, hi + 1 - (hi % 2))
        slabs[1] = (slabs[0][1], slabs[1][1])
    return slabs


def run_grid(ctx, pctype, dim, dims, opts, its, slab, B, S, b_full, y0_full):
    nx, ny, nz = dims
    base = pmg.Mat.laplace(ctx, dim, nx, ny, nz, kappa=1.0, slab=slab)
    nloc, _, row0 = base.size
    mat = pmg.Mat.lrc(base, B[row0:row0 + nloc], S)
    pc = pmg.PC(ctx, pctype)
    pc.set_operator(mat)
    pc.set_options(dict(opts, **{"-pc_b200_noise": "philox"}))
    pc.setup()
    ctx.set_seed(4242)
    y = y0_full[row0:row0 + nloc].copy()
    pc.apply_richardson(b_full[row0:row0 + nloc].copy(), y, its=its)
    return row0, y, ctx.draw_counter


def gather(parts, n):
    got = np.empty(n)
    for r0, yy in parts:
        got[r0:r0 + yy.size] = yy
    return got


def grid_case(ctx, rank, world, name):
    pctype, dim, dims, opts, its, ragged, k = CASES[name]
    slabs = slabs_for(dim, dims, world, ragged)
    n = dims[0] * dims[1] * dims[2]
    rng = np.random.default_rng(99)
    B, S = obs_matrix(rng, n, k), rng.uniform(20.0, 200.0, k)
    b_full, y0_full = rng.standard_normal(n), rng.standard_normal(n)
    row0, y, draws = run_grid(ctx, pctype, dim, dims, opts, its, slabs[rank], B, S, b_full, y0_full)
    _, y2, _ = run_grid(ctx, pctype, dim, dims, opts, its, slabs[rank], B, S, b_full, y0_full)
    parts = [None] * world
    dist.all_gather_object(parts, (row0, y, y2, draws))
    ok = True
    if rank == 0:
        got, got2 = gather([(p[0], p[1]) for p in parts], n), gather([(p[0], p[2]) for p in parts], n)
        single = pmg.Context(0, seed=4242)  # no communicator: the one-GPU path
        _, ref, ref_draws = run_grid(single, pctype, dim, dims, opts, its, None, B, S, b_full, y0_full)
        err = np.abs(got - ref).max() / np.abs(ref).max()
        rerun = np.array_equal(got, got2)
        counters = {p[3] for p in parts}
        ok = err <= TOL and rerun and counters == {ref_draws}
        print(f"[mgpu-lrc] {name}: world={world} slabs={slabs} k={k} max|d|/max|y|={err:.2e} rerun_bitwise={rerun} "
              f"draw_counters={sorted(counters)} single={ref_draws} -> {'OK' if ok else 'FAIL'}", flush=True)
        single.close()
    dist.barrier()
    return ok


def csr_case(ctx, rank, world):
    """Row-partitioned CSR base: the randomly permuted 2D Laplacian of mgpu_worker.csr_dist_case, uneven row starts."""
    import oracle as orc
    import scipy.sparse as sp
    A0 = orc.laplace(2, 33, 29, kappa=1.0)
    n, k = A0.n, 5
    rng = np.random.default_rng(7)
    perm = rng.permutation(n)
    M = sp.csr_matrix(A0.to_scipy())[perm][:, perm].tocsr()
    M.sort_indices()
    A = orc.CSR(n, M.indptr.astype(np.int64), M.indices.astype(np.int32), M.data.astype(np.float64))
    starts = np.round(np.linspace(0, n, world + 1) + (np.arange(world + 1) % 2) * 3).astype(np.int64)
    starts[0], starts[-1] = 0, n
    r0, r1 = int(starts[rank]), int(starts[rank + 1])
    B, S = obs_matrix(rng, n, k), rng.uniform(20.0, 200.0, k)
    rp = (M.indptr[r0:r1 + 1] - M.indptr[r0]).astype(np.int64)
    base = pmg.Mat.from_csr_dist(ctx, n, r0, rp, M.indices[M.indptr[r0]:M.indptr[r1]].astype(np.int64), M.data[M.indptr[r0]:M.indptr[r1]].astype(np.float64))
    mat = pmg.Mat.lrc(base, B[r0:r1], S)
    ncol, mycol = base.get_coloring()
    b_full, y0_full, x_full = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n)
    opts = {"-pc_mcgibbs_symmetric": "", "-pc_mcgibbs_omega": 1.2, "-pc_b200_noise": "philox"}
    pc = pmg.PC(ctx, "mcgibbs")
    pc.set_operator(mat)
    pc.set_options(opts)
    pc.setup()
    ctx.set_seed(4242)
    y = y0_full[r0:r1].copy()
    pc.apply_richardson(b_full[r0:r1].copy(), y, its=3)
    draws = ctx.draw_counter
    mc = pmg.MCSOR(mat)
    mc.set_omega(1.3)
    mc.set_sweep_type(3)
    ys = y0_full[r0:r1].copy()
    mc.apply(b_full[r0:r1].copy(), ys)
    ax = mat.mult(x_full[r0:r1].copy())
    parts = [None] * world
    dist.all_gather_object(parts, (r0, y, ys, ax, mycol, ncol, draws))
    ok = True
    if rank == 0:
        got, gots, gax = (gather([(p[0], p[i]) for p in parts], n) for i in (1, 2, 3))
        col = np.empty(n, np.int32)
        for p in parts:
            col[p[0]:p[0] + p[4].size] = p[4]
        kk = max(p[5] for p in parts)
        coloring = orc.Coloring(col, kk)
        single = pmg.Context(0, seed=4242)
        m1 = pmg.Mat.from_csr(single, A.rowptr, A.col, A.val)
        m1.set_coloring(col, kk)
        l1 = pmg.Mat.lrc(m1, B, S)
        p1 = pmg.PC(single, "mcgibbs")
        p1.set_operator(l1)
        p1.set_options(opts)
        p1.setup()
        single.set_seed(4242)
        ref = y0_full.copy()
        p1.apply_richardson(b_full.copy(), ref, its=3)
        Bb = {d: orc.lrc_build_correction(A, B, S, coloring, 1.0, d) for d in (orc.SOR_FORWARD, orc.SOR_BACKWARD)}
        refs = orc.lrc_mcsor_apply(A, B, Bb, b_full, y0_full.copy(), coloring, 1.3, orc.SOR_SYMMETRIC)
        refx = M @ x_full + B @ (S * (B.T @ x_full))
        e1 = np.abs(got - ref).max() / np.abs(ref).max()
        e2 = np.abs(gots - refs).max() / np.abs(refs).max()
        e3 = np.abs(gax - refx).max() / np.abs(refx).max()
        counters = {p[6] for p in parts}
        ok = e1 <= TOL and e2 <= TOL and e3 <= TOL and counters == {single.draw_counter}
        print(f"[mgpu-lrc] csr_dist: world={world} starts={starts.tolist()} sampler_vs_1gpu={e1:.2e} mcsor_vs_oracle={e2:.2e} "
              f"mult={e3:.2e} draw_counters={sorted(counters)} single={single.draw_counter} -> {'OK' if ok else 'FAIL'}", flush=True)
        single.close()
    dist.barrier()
    return ok


def posterior_mean_case(ctx, rank, world):
    """test_lrc_posterior_mean_device_rng on slabs: the sample mean approaches (A + B S B^T)^-1 b."""
    import oracle as orc
    dims = (17, 17)
    A = orc.laplace(2, *dims, kappa=3.0)
    n, k = A.n, 6
    rng = np.random.default_rng(20260625)
    B, S = obs_matrix(rng, n, k), np.full(k, 100.0)
    b = rng.standard_normal(n)
    slab = pmg.partition_slabs(dims[1], world, align=1)[rank]
    base = pmg.Mat.laplace(ctx, 2, *dims, kappa=3.0, slab=slab)
    nloc, _, row0 = base.size
    mat = pmg.Mat.lrc(base, B[row0:row0 + nloc], S)
    pc = pmg.PC(ctx, "mcgibbs")
    pc.set_operator(mat)
    pc.set_options({"-pc_mcgibbs_symmetric": "", "-pc_b200_noise": "philox"})
    pc.setup()
    ctx.set_seed(0xCAFE)
    y, acc, nsamp = np.zeros(nloc), np.zeros(nloc), 6000
    bl = b[row0:row0 + nloc].copy()
    pc.apply_richardson(bl, y, its=100)  # burn-in

    def cb(it, ys):
        acc[:] += ys

    pc.set_sample_callback(cb)
    pc.apply_richardson(bl, y, its=nsamp)
    parts = [None] * world
    dist.all_gather_object(parts, (row0, acc / nsamp))
    ok = True
    if rank == 0:
        got = gather(parts, n)
        mean = np.linalg.solve(A.to_scipy().toarray() + B @ np.diag(S) @ B.T, b)
        rel = np.linalg.norm(got - mean) / np.linalg.norm(mean)
        ok = rel < 0.1
        print(f"[mgpu-lrc] posterior_mean: world={world} |mean - (A + BSB^T)^-1 b| / |.| = {rel:.3f} -> {'OK' if ok else 'FAIL'}", flush=True)
    dist.barrier()
    return ok


def error_case(ctx, rank, world):
    """Refusals on a distributed low-rank operator fail on EVERY rank with the documented code, and nothing hangs."""
    dims = (33, 32)
    n, k = dims[0] * dims[1], 3
    rng = np.random.default_rng(5)
    B, S = obs_matrix(rng, n, k), rng.uniform(20.0, 200.0, k)
    slab = pmg.partition_slabs(dims[1], world)[rank]
    base = pmg.Mat.laplace(ctx, 2, *dims, kappa=1.0, slab=slab)
    nloc, _, row0 = base.size
    Bl = B[row0:row0 + nloc]
    codes = []
    mat = pmg.Mat.lrc(base, Bl, S)
    for pctype, opts in (("woodbury", {"-pc_woodbury_sampler": "mcgibbs", "-pc_woodbury_solver": "cholesky"}), ("cholsampler", {})):
        pc = pmg.PC(ctx, pctype)
        pc.set_operator(mat)
        pc.set_options(opts)
        try:
            pc.setup()
            codes.append(("%s accepted" % pctype, 0))
        except pmg.PMGError as e:
            codes.append((pctype, e.code))
    S_bad = S.copy()
    if rank == world - 1:
        S_bad[1] = np.nextafter(S_bad[1], np.inf)  # one ulp on one rank
    try:
        pmg.Mat.lrc(base, Bl, S_bad)
        codes.append(("S mismatch accepted", 0))
    except pmg.PMGError as e:
        codes.append(("S mismatch", e.code))
    # the communicator is still usable: a distributed product after the refusals
    x = rng.standard_normal(n)
    ax = mat.mult(x[row0:row0 + nloc].copy())
    parts = [None] * world
    dist.all_gather_object(parts, (row0, ax, codes))
    ok = True
    if rank == 0:
        got = gather([(p[0], p[1]) for p in parts], n)
        import oracle as orc
        refx = orc.laplace(2, *dims, kappa=1.0).to_scipy() @ x + B @ (S * (B.T @ x))
        e = np.abs(got - refx).max() / np.abs(refx).max()
        want = [("woodbury", 2), ("cholsampler", 2), ("S mismatch", 1)]
        ok = all(p[2] == want for p in parts) and e <= TOL
        print(f"[mgpu-lrc] errors: world={world} codes={[p[2] for p in parts]} mult_after={e:.2e} -> {'OK' if ok else 'FAIL'}", flush=True)
    dist.barrier()
    return ok


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = pmg.Context(local, seed=4242)
    uid = [pmg.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    ctx.comm_init(rank, world, uid[0])
    failed = []
    for name in sorted(CASES):
        if not grid_case(ctx, rank, world, name):
            failed.append(name)
    for name, fn in (("csr_dist", csr_case), ("posterior_mean", posterior_mean_case), ("errors", error_case)):
        if not fn(ctx, rank, world):
            failed.append(name)
    flag = torch.tensor([len(failed)], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(1 if int(flag.item()) else 0)


if __name__ == "__main__":
    main()
