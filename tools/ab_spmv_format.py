#!/usr/bin/env python
"""A/B of the SpMV storage inside cg! on one GPU: spmv_format 1 (CSR) against 0 (the offset-diagonal copy) on the
same operator, in one process.

For each grid (default 512 and 256): laplace_matrix(Float64, N, 3) is built once, both arms are warmed up, then the
arms alternate for --rounds rounds of --steps fixed-count cg! steps of --iters iterations each, every round timed with
the context's CUDA events between a barrier and a synchronise (as bench.py times its steps).  Then one more step per
arm with the per-kernel event brackets (b200_ctx_profile_*) gives the SpMV kernel's time, and the residual histories
and x of the two arms are compared bit for bit.

    python tools/ab_spmv_format.py [--grids 512 256] [--rounds 6] [--steps 10] [--iters 200] [--json out.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DATASHEET_HBM_GBS = 7700.0   # HGX B200 data sheet, one GPU


def gpu_facts():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else f"nvidia-smi failed: {out.stdout.strip()}"


def measured_hbm_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"])
    except (OSError, KeyError, ValueError):
        return None


def run_grid(isb, N, args):
    import torch
    ctx = isb.default_context()
    L = isb.lib()
    n = N ** 3
    A = isb.B200CSR.laplacian(N, 3)
    assert A.format == "dia", "the 7-point Laplacian must carry a DIA copy"
    b_host = np.random.default_rng(1234321).standard_normal(n)
    b_host /= np.sqrt(np.sum(b_host * b_host))
    b = isb.DeviceArray.from_numpy(ctx, b_host)
    x = isb.DeviceArray.zeros(ctx, n)
    out = {}

    def set_fmt(f):
        isb._lib.check(L.b200_ctx_set_option(ctx._h, b"spmv_format", f))

    def step():
        L.b200_fill(ctx._h, n, 0.0, x._p, 0)
        _, h = isb.cg_(x, A, b, initially_zero=True, maxiter=args.iters, reltol=0.0, _fixed_iterations=True, log=True)
        return h

    arms = {1: "csr", 0: "dia"}
    for f in arms:
        set_fmt(f)
        for _ in range(2):
            step()
    rates = {a: [] for a in arms.values()}
    for r in range(args.rounds):
        for f, a in arms.items():
            set_fmt(f)
            ctx.barrier()
            torch.cuda.synchronize()
            ctx.timer_start()
            for _ in range(args.steps):
                step()
            ms = ctx.timer_stop()
            ctx.barrier()
            torch.cuda.synchronize()
            rates[a].append(args.steps * args.iters / (ms / 1e3))
            print(f"N={N} round {r} {a}: {rates[a][-1]:.1f} it/s", flush=True)
    # kernel times (event brackets) and the outputs of one step per arm
    nnz = A.nnz
    bytes_k2 = {"csr": nnz * 12 + (n + 1) * 4 + 2 * n * 8, "dia": 7 * n * 8 + n + 2 * n * 8}
    results = {}
    for f, a in arms.items():
        set_fmt(f)
        L.b200_ctx_profile_enable(ctx._h, 1)
        for s in range(4):
            L.b200_ctx_profile_read(ctx._h, s, None, None, 1)
        h = step()
        torch.cuda.synchronize()
        prof = []
        for s in range(4):
            t, c = C.c_double(), C.c_int64()
            L.b200_ctx_profile_read(ctx._h, s, C.byref(t), C.byref(c), 1)
            prof.append(t.value / max(c.value, 1))
        L.b200_ctx_profile_enable(ctx._h, 0)
        results[a] = (np.asarray(h["resnorm"]).copy(), x.numpy().copy(), prof)
    set_fmt(0)
    peak = measured_hbm_gbs()
    for a in arms.values():
        v = np.asarray(rates[a])
        k2 = results[a][2][0]
        gbs = bytes_k2[a] / (k2 * 1e-3) / 1e9
        out[a] = {"its": [round(q, 2) for q in v], "median": float(np.median(v)), "min": float(v.min()),
                  "max": float(v.max()), "k2_ms": k2, "k1_ms": results[a][2][2], "k3_ms": results[a][2][1],
                  "k2_bytes": bytes_k2[a], "k2_gbs": gbs, "k2_frac_measured_peak": gbs / peak if peak else None,
                  "k2_frac_datasheet_7700": gbs / DATASHEET_HBM_GBS}
        print(f"N={N} {a}: median {out[a]['median']:.1f} it/s (min {out[a]['min']:.1f}, max {out[a]['max']:.1f}); "
              f"K2 {k2:.4f} ms, {bytes_k2[a] / 1e9:.3f} GB -> {gbs:.0f} GB/s "
              f"({'%.3f' % (gbs / peak) if peak else 'n/a'} of measured peak, {gbs / DATASHEET_HBM_GBS:.3f} of 7.7 TB/s)",
              flush=True)
    hc, xc, _ = results["csr"]
    hd, xd, _ = results["dia"]
    out["speedup_median"] = out["dia"]["median"] / out["csr"]["median"]
    out["slowest_dia_over_fastest_csr"] = out["dia"]["min"] / out["csr"]["max"]
    out["history_bitwise_equal"] = bool(hc.shape == hd.shape and np.array_equal(hc.view(np.int64), hd.view(np.int64)))
    out["x_bitwise_equal"] = bool(np.array_equal(xc.view(np.int64), xd.view(np.int64)))
    print(f"N={N}: dia/csr median {out['speedup_median']:.3f}x, slowest dia / fastest csr "
          f"{out['slowest_dia_over_fastest_csr']:.3f}; history bitwise equal {out['history_bitwise_equal']}, "
          f"x bitwise equal {out['x_bitwise_equal']}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, nargs="+", default=[512, 256])
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--json", default=None, help="also write the results here")
    args = ap.parse_args()
    import iterativesolvers_jl_b200 as isb
    res = {"gpu": gpu_facts(), "measured_hbm_gbs": measured_hbm_gbs(),
           "method": f"{args.rounds} alternating rounds per arm of {args.steps} x {args.iters}-iteration fixed-count "
                     "cg! steps, CUDA events between barrier + synchronise; K2 from b200_ctx_profile_* brackets of one "
                     "extra step; K2 bytes: CSR nnz*12 + (n+1)*4 + 2n*8, DIA 7n*8 + n + 2n*8"}
    print("gpu:", res["gpu"], flush=True)
    for N in args.grids:
        res[f"grid_{N}"] = run_grid(isb, N, args)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
