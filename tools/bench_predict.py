#!/usr/bin/env python3
"""Posterior prediction at grid scale: SVGPGibbs.predict (kernel by kernel from Python, T = K C stored per chunk) against
SVGPGibbs.predictive (npgp_svgp_predict_prepare + npgp_svgp_predict: one C call, no T).  Prints ONE JSON line with the device
name and power limit read in the same run.

  python tools/bench_predict.py [--reps 3] [--grid 4096]

  (a) rows/s of both paths on the bench leg c5 workload (4096 x 4096 lat/lon grid, diagonal Gibbs kernel, M = 1024, d = 2,
      trained-looking m, Ls as in bench_legs.leg_c5) and on a full-matrix d = 3 grid with as many rows (256^3), the two paths
      alternated `reps` times each in one process; the line gives every sample and the spread (max - min) / min
  (b) npgp_o8_rowquad_digits at 65536 x 1024 with and without T, CUDA events over 20 launches (3 alternating rounds)
  (c) parity of predictive against oracle.svgp_gibbs_predict on 4096 sampled grid rows (and against predict on all rows)"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
F64 = torch.float64
M = 1024


def device_info():
    info = {"device": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def rel(a, b):
    a, b = a.detach().double().cpu().reshape(-1), b.detach().double().cpu().reshape(-1)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def workload(variant, d, side):
    """Model with a trained-looking variational state (bench_legs.leg_c5) and the grid rows, both on cuda:0."""
    from bench import make_params
    from nonstationary_precip_b200.svgp import SVGPGibbs
    g = torch.Generator().manual_seed(5)
    kw = make_params(variant, M, d)
    kw["m"] = 0.3 * torch.randn(M, generator=g, dtype=F64)
    kw["Ls"] = 0.8 * torch.eye(M, dtype=F64) + 0.02 * torch.tril(torch.randn(M, M, generator=g, dtype=F64))
    Z = torch.rand(M, d, generator=g, dtype=F64) * 2 - 1
    dev = torch.device("cuda", 0)
    model = SVGPGibbs(variant, Z.to(dev), 1 << 20, **{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in kw.items()})
    lin = torch.linspace(-1, 1, side, dtype=F64, device=dev)
    xs = torch.stack(torch.meshgrid(*([lin] * d), indexing="ij"), -1).reshape(-1, d).contiguous()
    return model, xs, Z, kw


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def oracle_parity(model, xs, Z, kw, mean, var):
    from nonstationary_precip_b200.svgp import _inv_softplus
    from oracle import gibbs_oracle as o
    idx = torch.randperm(xs.shape[0], generator=torch.Generator().manual_seed(1))[:4096].to(xs.device)
    extra = (dict(log_ell_z=kw["log_ell_z"], prior_c=kw["prior_c"], prior_os=kw["prior_os"], prior_lam=kw["prior_lam"])
             if model.variant == "diag" else
             dict(H=kw["H"], Dm=kw["Dm"], row_os=torch.tensor(float(kw["row_os"]), dtype=F64), row_lam=kw["row_lam"]))
    mu_w, var_w = o.svgp_gibbs_predict(xs[idx].cpu(), Z, kw["m"], kw["Ls"], torch.tensor(_inv_softplus(kw["outputscale"]),
                                                                                         dtype=F64), model.variant, **extra)
    p = {"rows": 4096, "mean_rel": rel(mean[idx], mu_w), "var_rel": rel(var[idx], var_w), "tol": 1e-6}
    p["ok"] = bool(p["mean_rel"] <= 1e-6 and p["var_rel"] <= 1e-6)
    return p


def bench_workload(name, variant, d, side, reps):
    model, xs, Z, kw = workload(variant, d, side)
    n = xs.shape[0]
    paths = {"predict_py_chunk262144": lambda x: model.predict(x, chunk=1 << 18),
             "predictive_c_chunk65536": lambda x: model.predictive(x, chunk=65536)[:2],
             "predictive_c_chunk262144": lambda x: model.predictive(x, chunk=1 << 18)[:2]}
    for fn in paths.values():  # warm-up on a slice: plans, buffers, lazy attributes
        fn(xs[:1 << 18])
    rates, outs = {k: [] for k in paths}, {}
    for _ in range(reps):
        for k, fn in paths.items():  # alternated
            ms, out = timed(lambda: fn(xs))
            rates[k].append(n / ms * 1e3)
            outs[k] = out
    res = {"what": name, "rows": n, "M": M, "d": d,
           "rows_per_s": {k: [round(v) for v in r] for k, r in rates.items()},
           "spread": {k: round((max(r) - min(r)) / min(r), 4) for k, r in rates.items()},
           "c_over_py_median": round(sorted(rates["predictive_c_chunk65536"])[reps // 2] /
                                     sorted(rates["predict_py_chunk262144"])[reps // 2], 4)}
    mean_c, var_c = outs["predictive_c_chunk65536"]
    mean_p, var_p = outs["predict_py_chunk262144"]
    res["c_vs_py_all_rows"] = {"mean_rel": rel(mean_c, mean_p), "var_rel": rel(var_c, var_p)}
    res["finite"] = bool(torch.isfinite(mean_c).all() and torch.isfinite(var_c).all())
    res["parity"] = oracle_parity(model, xs, Z, kw, mean_c, var_c)
    del model, xs, outs
    torch.cuda.empty_cache()
    return res


def bench_rowquad(rounds=3, launches=20):
    from nonstationary_precip_b200 import ops
    n, d = 65536, 2
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
    Cm = A @ A.T / M - 0.3 * torch.eye(M, dtype=F64, device=dev)
    Cm = 0.5 * (Cm + Cm.T)
    Cd = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device=dev)
    cexp = torch.empty(M, dtype=torch.int32, device=dev)
    ops.o8_slice_rows(Cm, 64, Cd, cexp)
    T = torch.empty(n, M, dtype=F64, device=dev)
    q1, q2 = torch.empty(M // 64, n, dtype=F64, device=dev), torch.empty(M // 64, n, dtype=F64, device=dev)
    runs = {"with_T": lambda: ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, T, q_part=q1),
            "without_T": lambda: ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, None, q_part=q2)}
    for fn in runs.values():
        fn()
    ms = {k: [] for k in runs}
    for _ in range(rounds):
        for k, fn in runs.items():
            t, _ = timed(lambda: [fn() for _ in range(launches)])
            ms[k].append(round(t / launches, 4))
    torch.cuda.synchronize()
    return {"what": "npgp_o8_rowquad_digits, %d x %d, q partials, CUDA events over %d launches per sample" % (n, M, launches),
            "ms_per_launch": ms, "T_bytes": n * M * 8, "q_bitwise_equal": bool(torch.equal(q1, q2))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--grid", type=int, default=4096, help="side of the 2-D grid; the 3-D grid has as many rows")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_predict.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = device_info()
    side3 = round(args.grid ** (2 / 3))
    out["rowquad"] = bench_rowquad()
    out["c5_diag_d2"] = bench_workload("c5: %dx%d grid, diagonal Gibbs SVGP, M=%d, d=2" % (args.grid, args.grid, M), "diag", 2,
                                       args.grid, args.reps)
    out["full_d3"] = bench_workload("%d^3 grid, full-matrix Gibbs SVGP, M=%d, d=3" % (side3, M), "full", 3, side3, args.reps)
    out["parity_ok"] = bool(out["c5_diag_d2"]["parity"]["ok"] and out["full_d3"]["parity"]["ok"] and
                            out["rowquad"]["q_bitwise_equal"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
