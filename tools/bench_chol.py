"""Times the dense Cholesky sampler (PCCHOLSAMPLER) across the 4096-unknown switch between its two paths.

usage: bench_chol.py [--sizes 4096,8192,16384,32768] [--out FILE.json]

n = 4096 runs the host-factor path (two dense n x n copies of W = L^-1); above 4096 the factor is formed on the device and
W's lower triangle is packed in 64 x 64 tiles.  Per size: set-up time (host clock around PCSetUp, which ends in a device
synchronise), time per sample from CUDA events over at least 1 s of back-to-back single samples (v = W b + z, y = W^T v),
and the time of one step of a chain (its > 1: the cached W b, then one product W^T (v + z)).  Compulsory traffic is one
read of the triangle per product, 8 n^2 bytes per sample; `bytes_streamed` counts what the packed tiles really hold
(diagonal tiles in full).  Bandwidth is given as a fraction of the 6539.9 GB/s device-to-device copy rate DESIGN.md §3
measured.  The operator is the 2D shifted Laplacian kappa^2 I + h L of src/problems.c (kappa = 1) on an nx x ny grid.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sp
import torch

import parmgmc_b200 as pmg

COPY_GBS = 6539.9
L2_BYTES = 126e6
GRIDS = {4096: (64, 64), 8192: (128, 64), 16384: (128, 128), 32768: (256, 128)}


def laplace2d(nx, ny, kappa=1.0):
    def t(m):
        deg = np.full(m, 2.0)
        deg[0] = deg[-1] = 1.0
        return sp.diags([-np.ones(m - 1), deg, -np.ones(m - 1)], [-1, 0, 1], format="csr")
    h = 1.0 / ((max(nx, ny) - 1) ** 2)
    A = (kappa ** 2 * sp.identity(nx * ny) + h * (sp.kron(sp.identity(ny), t(nx)) + sp.kron(t(ny), sp.identity(nx)))).tocsr()
    A.sort_indices()
    return A


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return name, pl


def timed(stream, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn(reps)
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def bench(ctx, stream, n):
    nx, ny = GRIDS.get(n, (n, 1))
    A = laplace2d(nx, ny)
    mat = pmg.Mat.from_csr(ctx, A.indptr.astype(np.int64), A.indices.astype(np.int32), A.data)
    pc = pmg.PC(ctx, "cholsampler")
    pc.set_operator(mat)
    pc.set_option("-pc_b200_noise", "philox")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pc.setup()
    setup_s = time.perf_counter() - t0
    view = pc.view()
    b = torch.randn(n, dtype=torch.float64, device="cuda")
    y = torch.zeros(n, dtype=torch.float64, device="cuda")

    def singles(k):
        for _ in range(k):
            pc.apply_richardson_dev(b, y, its=1)

    def chain(k):
        pc.apply_richardson_dev(b, y, its=k)

    singles(20)  # warm-up
    chain(20)
    torch.cuda.synchronize()
    est = timed(stream, singles, 20) / 20
    reps = max(200, int(1.0 / est) + 1)
    t_sample = timed(stream, singles, reps) / reps
    t_chain = timed(stream, chain, reps) / reps
    nt = (n + 63) // 64
    packed = n > 4096
    tri_bytes = nt * (nt + 1) // 2 * 64 * 64 * 8 if packed else 8 * n * (n + 1) // 2  # bytes one product reads
    compulsory = 8.0 * n * n
    res = {
        "n": n, "grid": [nx, ny], "path": "device factor, packed triangle" if packed else "host factor, two dense copies",
        "setup_s": round(setup_s, 4),
        "sample_us": round(t_sample * 1e6, 2), "samples_timed": reps, "chain_step_us": round(t_chain * 1e6, 2),
        "bytes_per_sample": compulsory, "bytes_streamed": 2.0 * tri_bytes,
        "sample_GBs": round(compulsory / t_sample / 1e9, 1),
        "fraction_of_copy_bw": round(compulsory / t_sample / 1e9 / COPY_GBS, 3),
        "chain_step_fraction_of_copy_bw": round(compulsory / 2 / t_chain / 1e9 / COPY_GBS, 3),
        "triangle_bytes": tri_bytes, "triangle_fits_l2": tri_bytes <= L2_BYTES,
        "view": view.strip().splitlines(),
    }
    pc.close()
    mat.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,8192,16384,32768")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_chol.py needs a CUDA device")
    stream = torch.cuda.current_stream()
    ctx = pmg.Context(0, stream=stream.cuda_stream, seed=0xCAFE)
    name, power = card()
    out = {"device": name, "power_limit": power, "copy_GBs_reference": COPY_GBS, "results": []}
    for n in [int(s) for s in args.sizes.split(",")]:
        r = bench(ctx, stream, n)
        print(json.dumps(r), flush=True)
        out["results"].append(r)
    ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
