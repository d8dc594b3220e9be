#!/usr/bin/env python3
"""Posterior sample fields at grid scale: SVGPGibbs.sample (npgp_svgp_predict_prepare + npgp_svgp_sample_prepare +
npgp_svgp_sample) against SVGPGibbs.predictive on the same rows.  Prints ONE JSON line with the device name and power limit
read in the same run.

  python tools/bench_sample.py [--reps 3] [--grid 4096]

  (a) on the workloads of tools/bench_predict.py (c5: 4096 x 4096 grid, diagonal Gibbs kernel, d = 2; a 256^3 grid with the
      full-matrix kernel, d = 3; M = 1024; 65536-row chunks): rows/s and draws/s (whole-grid fields per second) of sample for
      S = 16 and S = 64, alternated with predictive `reps` times each in one process; every sample and the spread
  (b) the new T-only contraction npgp_o8_gemm_digits at 65536 x S_pad x 1024 next to the q-only row-quadratic pass
      (npgp_o8_rowquad_digits, T = NULL) at 65536 x 1024, CUDA events over 20 launches (3 alternating rounds)"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_predict import F64, M, device_info, rel, timed, workload  # noqa: E402

CHUNK = 65536
SAMPLES = (16, 64)


def bench_workload(name, variant, d, side, reps):
    model, xs, Z, kw = workload(variant, d, side)
    n = xs.shape[0]
    paths = {"predictive": lambda x: model.predictive(x, chunk=CHUNK).mean}
    for S in SAMPLES:
        paths["sample_S%d" % S] = lambda x, S=S: model.sample(x, S, seed=1, chunk=CHUNK)
    for fn in paths.values():  # warm-up on a slice: plans, buffers, lazy attributes
        fn(xs[:1 << 18])
    ms, outs = {k: [] for k in paths}, {}
    for _ in range(reps):
        for k, fn in paths.items():  # alternated
            t, out = timed(lambda: fn(xs))
            ms[k].append(t)
            outs[k] = out
    res = {"what": name, "rows": n, "M": M, "d": d, "chunk": CHUNK,
           "rows_per_s": {k: [round(n / t * 1e3) for t in v] for k, v in ms.items()},
           "spread": {k: round((max(v) - min(v)) / min(v), 4) for k, v in ms.items()}}
    res["draws_per_s"] = {k: [round(int(k[8:]) / t * 1e3, 3) for t in ms[k]] for k in ms if k.startswith("sample_S")}
    med = {k: sorted(v)[reps // 2] for k, v in ms.items()}
    res["sample_over_predictive_time_median"] = {k: round(med[k] / med["predictive"], 4) for k in ms if k != "predictive"}
    mean = outs["predictive"]
    res["finite"] = bool(all(torch.isfinite(o).all() for o in outs.values()))
    # the mean of the 64 draws over the grid, in standard errors of the average of 64 draws of var_f
    var = model.predictive(xs, chunk=CHUNK).var
    z = (outs["sample_S64"].mean(0) - mean).abs() / torch.sqrt(var / 64)
    res["S64_average_minus_mean_in_se"] = {"max": round(z.max().item(), 3), "rms": round(z.pow(2).mean().sqrt().item(), 4)}
    # separate prepares: at M >= 512 the M x M products of the prepares add split-K partials with FP64 atomics, so draws of
    # two calls agree to rounding rather than bitwise
    a, b = outs["sample_S16"], outs["sample_S64"][:16]
    res["S16_vs_first_16_of_S64"] = {"bitwise": bool(torch.equal(a, b)), "max_rel": rel(a, b)}
    del model, xs, outs, var, z, a, b
    torch.cuda.empty_cache()
    return res


def bench_kernels(rounds=3, launches=20):
    from nonstationary_precip_b200 import ops
    from nonstationary_precip_b200._lib import check, lib
    n, d = CHUNK, 2
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(3)
    x = (torch.rand(n, d, generator=g, dtype=F64) * 2 - 1).to(dev)
    z = (torch.rand(M, d, generator=g, dtype=F64) * 2 - 1).to(dev)
    ex = torch.exp(0.3 * torch.randn(d, n, generator=g, dtype=F64) - 1.0).to(dev)
    ez = torch.exp(0.3 * torch.randn(d, M, generator=g, dtype=F64) - 1.0).to(dev)
    s = torch.tensor([0.644], dtype=F64, device=dev)
    digits = torch.empty(ops.digits_bytes(n, M, 128), dtype=torch.uint8, device=dev)
    ops.gibbs_diag_fwd_digits(x, ex, z, ez, s, digits)
    A = torch.randn(M, M, generator=g, dtype=F64).to(dev)
    G = A @ A.T / M
    Gd = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device=dev)
    gexp = torch.empty(M, dtype=torch.int32, device=dev)
    ops.o8_slice_rows(G, 64, Gd, gexp)
    q = torch.empty(M // 64, n, dtype=F64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    runs = {"rowquad_q_only_%dx%d" % (n, M): lambda: ops.o8_rowquad_digits(n, M, digits, s, Gd, gexp, None, q_part=q)}
    for Sp in SAMPLES:
        Sp = (Sp + 63) // 64 * 64
        Wt = torch.randn(Sp, M, generator=g, dtype=F64).to(dev)
        Wd = torch.empty(ops.digits_bytes(Sp, M, 64), dtype=torch.uint8, device=dev)
        wexp = torch.empty(Sp, dtype=torch.int32, device=dev)
        ops.o8_slice_rows(Wt, 64, Wd, wexp)
        F = torch.empty(n, Sp, dtype=F64, device=dev)
        runs.setdefault("gemm_digits_%dx%dx%d" % (n, Sp, M), lambda Sp=Sp, Wd=Wd, wexp=wexp, F=F: check(
            lib().npgp_o8_gemm_digits(n, Sp, M, digits.data_ptr(), None, s.data_ptr(), Wd.data_ptr(), wexp.data_ptr(),
                                      F.data_ptr(), Sp, st), "npgp_o8_gemm_digits"))
    for fn in runs.values():
        fn()
    ms = {k: [] for k in runs}
    for _ in range(rounds):
        for k, fn in runs.items():
            t, _ = timed(lambda: [fn() for _ in range(launches)])
            ms[k].append(round(t / launches, 4))
    torch.cuda.synchronize()
    return {"what": "digit contractions on one %d-row chunk, CUDA events over %d launches per sample" % (n, launches),
            "ms_per_launch": ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--grid", type=int, default=4096, help="side of the 2-D grid; the 3-D grid has as many rows")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_sample.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = device_info()
    side3 = round(args.grid ** (2 / 3))
    out["kernels"] = bench_kernels()
    out["c5_diag_d2"] = bench_workload("c5: %dx%d grid, diagonal Gibbs SVGP, M=%d, d=2" % (args.grid, args.grid, M), "diag", 2,
                                       args.grid, args.reps)
    out["full_d3"] = bench_workload("%d^3 grid, full-matrix Gibbs SVGP, M=%d, d=3" % (side3, M), "full", 3, side3, args.reps)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
