#!/usr/bin/env python3
"""Posterior of regional sums at scale: SVGPGibbs.region_posterior (npgp_svgp_predict_prepare + npgp_svgp_region_moments) and
its pair-sum kernel alone (npgp_gibbs_*_segsum), next to the per-pair rate of the forward digit kernel
(npgp_gibbs_*_fwd_digits) on the same variant and d.  Prints ONE JSON line with the device name and power limit read in the
same run.

  python tools/bench_region.py [--reps 2]

  workloads (M = 1024, rows of the grids of tools/bench_predict.py, 65536-row chunks): variant 1 (full-matrix kernel, d = 3)
  and variant 0 (diagonal kernel, d = 2); n in {2^16, 2^18, 2^20} rows in R in {1, 64, 1024} equal regions of consecutive
  grid rows; variances only (sum_r n_r (n_r - 1) / 2 pairs) and the full covariance (n (n - 1) / 2 pairs).  Per case: ms of
  the whole call and of the pair sums alone (CUDA events, `reps` samples, the pair sums alternated with the call), pairs/s of
  the pair sums.  The digit kernel: 65536 x 1024, CUDA events over 20 launches."""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_predict import M, device_info, timed, workload  # noqa: E402

CHUNK = 65536
NS = (1 << 16, 1 << 18, 1 << 20)
RS = (1, 64, 1024)


def digits_rate(model, xs, field, launches=20):
    from nonstationary_precip_b200 import ops
    n = 65536
    x, s = xs[:n].contiguous(), torch.nn.functional.softplus(model.p["raw_outputscale"])
    digits = torch.empty(ops.digits_bytes(n, M, 128), dtype=torch.uint8, device=xs.device)
    fz = model._field_z()
    if model.variant == "full":
        f = lambda: ops.gibbs_full_fwd_digits(x, field[:n].contiguous(), model.p["Z"], fz, 1e-5, s, digits)
    else:
        f = lambda: ops.gibbs_diag_fwd_digits(x, field[:, :n].contiguous(), model.p["Z"], fz, s, digits)
    f()
    ms = [timed(lambda: [f() for _ in range(launches)])[0] / launches for _ in range(3)]
    return {"ms": [round(t, 4) for t in ms], "pairs_per_s": round(n * M / min(ms) * 1e3)}


def bench(variant, d, side, reps):
    from nonstationary_precip_b200 import ops
    from nonstationary_precip_b200.svgp import region_segments
    model, grid, _, _ = workload(variant, d, side)
    grid = grid[:NS[-1]].contiguous()
    field_all = model.predictive(grid, field=True, chunk=CHUNK).field
    s = torch.nn.functional.softplus(model.p["raw_outputscale"])
    out = {"variant": 1 if variant == "full" else 0, "d": d, "M": M, "digits_fwd": digits_rate(model, grid, field_all)}
    cases = []
    for n in NS:
        xs = grid[:n].contiguous()
        fld = field_all[:n].contiguous() if variant == "full" else field_all[:, :n].contiguous()
        for R in RS:
            labels = torch.arange(n, device=xs.device) * R // n
            _, seg = region_segments(labels, R)
            nr = torch.bincount(labels, minlength=R).double()
            for cov in (False, True):
                pairs = int((nr * (nr - 1) / 2).sum().item()) if not cov else n * (n - 1) // 2
                if variant == "full":
                    pair = lambda: ops.gibbs_full_segsum(xs, fld, seg, full=cov, scale=s)
                else:
                    pair = lambda: ops.gibbs_diag_segsum(xs, fld, seg, full=cov, scale=s)
                call = lambda: model.region_posterior(xs, labels, R, cov=cov, chunk=CHUNK)
                k = 1 if pairs > 1e11 else reps
                if pairs < 1e10:  # warm-up: plans, buffers (the largest cases follow smaller ones of the same shapes)
                    pair(), call()
                t_pair, t_call = [], []
                for _ in range(k):
                    t_pair.append(timed(pair)[0])
                    t, r = timed(call)
                    t_call.append(t)
                cases.append({"n": n, "R": R, "cov": cov, "pairs": pairs, "ms_call": [round(t, 3) for t in t_call],
                              "ms_pairs": [round(t, 3) for t in t_pair],
                              "pairs_per_s": round(pairs / min(t_pair) * 1e3) if pairs else None,
                              "finite": bool(torch.isfinite(r.var).all() and torch.isfinite(r.mean).all())})
    out["cases"] = cases
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_region.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"tool": "bench_region", **device_info(),
           "workloads": [bench("full", 3, 102, args.reps), bench("diag", 2, 1024, args.reps)]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
