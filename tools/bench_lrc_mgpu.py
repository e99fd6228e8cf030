"""Low-rank-corrected samplers (MATLRC, BASELINE config 5's observation term) weak-scaled over N GPUs.
usage: python -m torch.distributed.run --nproc-per-node N tools/bench_lrc_mgpu.py [--out FILE] [--n 4097] [--k 17] [--samples S]

Geometry of bench.py: one n x (n-1) slab per rank, the last rank owning the closing row (n x n on one GPU).  k disc-shaped
observation columns (weight 1 inside a disc of radius 12 nodes) spread over the global grid.  For mcgibbs (symmetric) and
gamgmc (default levels), with and without the low-rank term: ms per sample (CUDA events, max over ranks), the low-rank share
(with minus without), the time of the lrc_* kernels and of the NCCL kernels per sample (torch.profiler, separate run), the
compulsory bytes of the low-rank streams (3 n_local k 8 B per directional sweep, 2 n_local k 8 B per residual) and the set-up
time.  Rank 0 prints one JSON line per configuration and writes them all to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import parmgmc_b200 as pmg  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=4097)
ap.add_argument("--k", type=int, default=17)
ap.add_argument("--samples", type=int, default=20)
ap.add_argument("--out", default="")
args = ap.parse_args()

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
stream = torch.cuda.current_stream()
ctx = pmg.Context(local, stream=stream.cuda_stream, seed=0xCAFE)
if world > 1:
    uid = [pmg.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    ctx.comm_init(rank, world, uid[0])

nx = args.n
ny = nx if world == 1 else (nx - 1) * world + 1
slab = pmg.partition_slabs(ny, world)[rank] if world > 1 else None
base = pmg.Mat.laplace(ctx, 2, nx, ny, kappa=1.0, slab=slab)
nloc, nglob, row0 = base.size
k = args.k

# disc observations: centres on a regular pattern over the global grid, rows of this rank only (column-major)
Bt = np.zeros((k, nloc))
r_disc = 12
gy0 = row0 // nx
rows_here = nloc // nx
cols = np.arange(nx)
for j in range(k):
    cx = int((j % 5 + 0.5) * nx / 5)
    cy = int((j // 5 + 0.5) * ny / ((k + 4) // 5))
    for gy in range(max(cy - r_disc, gy0), min(cy + r_disc + 1, gy0 + rows_here)):
        inside = (cols - cx) ** 2 + (gy - cy) ** 2 <= r_disc * r_disc
        Bt[j, (gy - gy0) * nx + cols[inside]] = 1.0
S = np.full(k, 1.0 / 0.01**2)  # sigma = 0.01


def max_over_ranks(v):
    t = torch.tensor([v], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def measure(pctype, lrc):
    opts = {"-pc_b200_noise": "philox"}
    if pctype == "mcgibbs":
        opts["-pc_mcgibbs_symmetric"] = ""
    barrier()
    t0 = time.perf_counter()
    mat = pmg.Mat.lrc(base, Bt.T, S) if lrc else base
    pc = pmg.PC(ctx, pctype)
    pc.set_operator(mat)
    pc.set_options(opts)
    pc.setup()
    y = torch.zeros(nloc, dtype=torch.float64, device="cuda")
    b = torch.zeros(nloc, dtype=torch.float64, device="cuda")
    pc.apply_richardson_dev(b, y, its=1)  # the low-rank corrections are built on the first sweep
    barrier()
    setup_s = max_over_ranks(time.perf_counter() - t0)
    pc.apply_richardson_dev(b, y, its=3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    pc.apply_richardson_dev(b, y, its=args.samples)
    e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.samples)
    # kernel times in a separate, profiled run
    from torch.profiler import ProfilerActivity, profile
    nprof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pc.apply_richardson_dev(b, y, its=nprof)
        barrier()
    lrc_us = nccl_us = 0.0
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name
        dur = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        if "lrc_" in name:
            lrc_us += dur
        elif "nccl" in name.lower():
            nccl_us += dur
    lrc_us, nccl_us = max_over_ranks(lrc_us / nprof), max_over_ranks(nccl_us / nprof)
    if pctype == "mcgibbs":
        streams_b = 2 * 3 * nloc * k * 8 if lrc else 0
    else:
        L = pc.gamgmc_get_levels()
        streams_b = sum((2 * 3 + 2) * pc.gamgmc_level_info(lv)[0] * k * 8 for lv in range(1, L)) if lrc else 0
    del pc
    return {"ms_per_sample": ms, "setup_s": setup_s, "lrc_kernel_us_per_sample": lrc_us, "nccl_kernel_us_per_sample": nccl_us,
            "lrc_compulsory_bytes_per_sample": streams_b}


card = ""
if rank == 0:
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[local]
    except Exception as e:  # noqa: BLE001
        card = f"nvidia-smi unavailable: {e}"
rows = []
for pctype in ("mcgibbs", "gamgmc"):
    off = measure(pctype, False)
    on = measure(pctype, True)
    share_ms = on["ms_per_sample"] - off["ms_per_sample"]
    row = {"n_gpus": world, "sampler": pctype + (" symmetric" if pctype == "mcgibbs" else " default levels"), "grid_global": [nx, ny], "n_local": nloc, "k": k,
           "ms_per_sample_without_lrc": round(off["ms_per_sample"], 4), "ms_per_sample_with_lrc": round(on["ms_per_sample"], 4),
           "lrc_share_ms": round(share_ms, 4), "lrc_kernels_ms": round(on["lrc_kernel_us_per_sample"] / 1e3, 4),
           "lrc_compulsory_GB_per_sample": round(on["lrc_compulsory_bytes_per_sample"] / 1e9, 3),
           "lrc_share_GB_per_s": round(on["lrc_compulsory_bytes_per_sample"] / (share_ms * 1e-3) / 1e9, 1) if share_ms > 0 else None,
           "lrc_kernels_GB_per_s": round(on["lrc_compulsory_bytes_per_sample"] / on["lrc_kernel_us_per_sample"] / 1e3, 1) if on["lrc_kernel_us_per_sample"] > 0 else None,
           "allgather_share_ms": round((on["nccl_kernel_us_per_sample"] - off["nccl_kernel_us_per_sample"]) / 1e3, 4),
           "setup_s_with_lrc": round(on["setup_s"], 2), "setup_s_without_lrc": round(off["setup_s"], 2), "card": card}
    rows.append(row)
    if rank == 0:
        print(json.dumps(row), flush=True)
if rank == 0 and args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rows, f, indent=1)
if world > 1:
    dist.destroy_process_group()
