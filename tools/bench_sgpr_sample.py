#!/usr/bin/env python3
"""Posterior sample fields of the streamed SGPR models at scale: posterior().sample() against posterior().predictive() on the
same snapshot.  Prints ONE JSON line with the device name and power limit read in the same run.

  python tools/bench_sgpr_sample.py [--reps 3] [--grid 4096] [--train 1048576] [--st-rows 1048576]

  (a) diagonal model (SGPRGibbsStream), M = 1024, d = 2, on the c5 grid (grid x grid rows on [-1, 1]^2, 65536-row chunks):
      rows/s and draws/s of sample() at S = 16 and 64, alternated with predictive(), `reps` samples each; the preparation
      (E^T, W^T = E^T V and its planes: sample() at one row); CUDA events over 20 launches of the two kernels sample() adds
      per 65536-row chunk, the contraction F = K W (npgp_o8_gemm_digits, S = 64) and the finisher (npgp_sgpr_sample_finish),
      next to the triangular pass against P it shares with predictive()
  (b) spatio-temporal model (SGPRSpatioTemporalStream), M = 2048 (feature width 4096), on `st-rows` c3-shaped rows: as (a)
      without the kernel times
The models are those of tools/bench_sgpr_predict.py."""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_predict import device_info, timed  # noqa: E402
from bench_sgpr_predict import diag_model, st_model, st_rows  # noqa: E402

F64 = torch.float64
CHUNK = 65536


def alternate(post, xs, reps):
    """predictive and sample (S = 16, 64) alternated on one snapshot; ms per call."""
    n = xs.shape[0]
    post.predictive(xs[:CHUNK + 1000], chunk=CHUNK)  # warm-up: both chunk shapes, every path
    for S in (16, 64):
        post.sample(xs[:CHUNK + 1000], S, chunk=CHUNK)
    ms = {"predictive": [], "sample_16": [], "sample_64": []}
    for _ in range(reps):
        ms["predictive"].append(timed(lambda: post.predictive(xs, chunk=CHUNK))[0])
        for S in (16, 64):
            t, out = timed(lambda: post.sample(xs, S, seed=7, chunk=CHUNK))
            ms["sample_%d" % S].append(t)
            finite = bool(torch.isfinite(out).all())
            del out
            assert finite
    res = {"rows": n, "ms": {k: [round(t, 1) for t in v] for k, v in ms.items()},
           "rows_per_s": {k: [round(n / t * 1e3) for t in v] for k, v in ms.items()},
           "draws_per_s": {k: [round(int(k[7:]) / t * 1e3, 2) for t in v] for k, v in ms.items() if k != "predictive"}}
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    res["sample_64_over_predictive_median"] = round(med(ms["sample_64"]) / med(ms["predictive"]), 3)
    post.sample(xs[:1], 64)
    res["prepare_ms_S64"] = [round(timed(lambda: post.sample(xs[:1], 64))[0], 2) for _ in range(3)]
    return res


def kernel_times(post, xs):
    """Per-launch ms of npgp_o8_gemm_digits (F = K W, S = 64), npgp_sgpr_sample_finish and the P pass on one chunk."""
    from nonstationary_precip_b200 import ops
    W, S = post.width, 64
    xc = xs[:CHUNK].contiguous()
    b = post._row_buffers(xc, CHUNK)
    mean = torch.empty(CHUNK, dtype=F64, device="cuda")
    post._row_chunk(b, 0, CHUNK, mean)
    Wt = ops.dgemm(ops.sample_normals(W, S, 7, torch.empty(S, W, dtype=F64, device="cuda")), post.V, tri_b=1)
    Wd = torch.empty(ops.digits_bytes(S, W, 64), dtype=torch.uint8, device="cuda")
    We = torch.empty(S, dtype=torch.int32, device="cuda")
    ops.o8_slice_rows(Wt, 64, Wd, We)
    Fc = torch.empty(CHUNK, S, dtype=F64, device="cuda")
    out = torch.empty(S, CHUNK, dtype=F64, device="cuda")
    fns = {"gemm_digits_65536x64": lambda: ops.o8_gemm_digits(CHUNK, S, W, b["Ad"], post.one, Wd, We, Fc),
           "finish_65536x64": lambda: ops.sgpr_sample_finish(mean, b["qn"], 0, Fc, S, post.s, post.noise, out),
           "trinorm_P_65536": lambda: ops.o8_trinorm_digits(CHUNK, W, W, b["Ad"], post.one, *post.planes[0], b["qn"])}
    res = {k: [] for k in fns}
    for _ in range(3):
        for k, fn in fns.items():
            fn()
            t, _ = timed(lambda: [fn() for _ in range(20)])
            res[k].append(round(t / 20, 4))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--grid", type=int, default=4096)
    ap.add_argument("--train", type=int, default=1 << 20)
    ap.add_argument("--st-rows", type=int, default=1 << 20)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    out = device_info()

    model, x, y = diag_model(a.train)
    side = torch.linspace(-1, 1, a.grid, dtype=F64, device="cuda")
    xs = torch.stack(torch.meshgrid(side, side, indexing="ij"), -1).reshape(-1, 2).contiguous()
    post = model.posterior(x, y, chunk=65536)
    out["diag_c5"] = dict(M=post.M, width=post.width, digits=post.digits, **alternate(post, xs, a.reps))
    out["diag_c5_kernels_ms"] = kernel_times(post, xs)
    del model, post, x, y, xs
    torch.cuda.empty_cache()

    model, x, y = st_model(a.train)
    xs = st_rows(a.st_rows, torch.Generator().manual_seed(4)).cuda()
    post = model.posterior(x, y, chunk=32768)
    out["st_c3"] = dict(M=post.M, width=post.width, digits=post.digits, **alternate(post, xs, a.reps))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
