#!/usr/bin/env python3
"""Grid-scale posterior of the exact Gibbs GP (DiagonalExactGP.posterior()): predictive() and sample() on a grid x grid map
of [-1, 1]^2.  Prints ONE JSON line with the device name and power limit read in the same run.

  python tools/bench_exact_posterior.py [--reps 3] [--grid 4096]

For each case, with 65536-row chunks: posterior() time; rows/s of predictive() and of sample() at S = 16 and 64, alternated,
`reps` calls each; the digit path against the FP64 path (use_i8 = False) on 65536 rows sampled from the grid (max relative
difference of mean, var and of 16 draws).  Cases: config 1's size, n = 316 training rows (d = 2), with no knots and with a
32 x 32 grid of knots (1024), and n = 4096 training rows with no knots.  The training rows are uniform on [-1, 1]^2 with
lengthscales 0.1 exp(0.2 N(0, 1)), y = sin(3 x_0) + 0.1 N(0, 1), outputscale 0.644 and noise 0.011 as in the experiment."""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_predict import device_info, timed  # noqa: E402

F64 = torch.float64
CHUNK = 65536


def exact_model(n, seed=0):
    from nonstationary_precip_b200.gp_base import GaussianLikelihood
    from nonstationary_precip_b200.models.gibbs_kernels import LogNormalPriorProcess
    from nonstationary_precip_b200.models.nonstationary_models import DiagonalExactGP
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 2, generator=g, dtype=F64) * 2 - 1
    y = torch.sin(3 * x[:, 0]) + 0.1 * torch.randn(n, generator=g, dtype=F64)
    prior = LogNormalPriorProcess(input_dim=2).cuda().double()
    prior.covar_module.outputscale = torch.ones_like(prior.covar_module.outputscale)
    prior.covar_module.base_kernel.lengthscale = 1.3 * torch.ones_like(prior.covar_module.base_kernel.lengthscale)
    prior.mean_module.constant = torch.nn.Parameter(math.log(0.3) * torch.ones_like(prior.mean_module.constant))
    for p in prior.parameters():
        p.requires_grad = False
    model = DiagonalExactGP(x.cuda(), y.cuda(), GaussianLikelihood().cuda().double(), prior, num_dim=2).cuda().double()
    model.likelihood.noise = 0.011
    model.covar_module.outputscale = 0.644
    with torch.no_grad():
        model.log_ell_train_x.copy_(math.log(0.1) + 0.2 * torch.randn(2, n, generator=g, dtype=F64))
    return model


def rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def case(model, knots, xs, reps):
    n = xs.shape[0]
    model.use_i8 = True
    t_post = [round(timed(lambda: model.posterior(knots=knots))[0], 1) for _ in range(3)]
    post = model.posterior(knots=knots)
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
    res = {"width": post.width, "digits": post.digits, "posterior_ms": t_post, "rows": n,
           "rows_per_s": {k: [round(n / t * 1e3) for t in v] for k, v in ms.items()}}
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(1))[:CHUNK].cuda()
    xr = xs[idx].contiguous()
    a, da = post.predictive(xr, chunk=CHUNK), post.sample(xr, 16, seed=3, chunk=CHUNK)
    del post
    model.use_i8 = False
    ref = model.posterior(knots=knots)
    b, db = ref.predictive(xr, chunk=CHUNK), ref.sample(xr, 16, seed=3, chunk=CHUNK)
    res["digits_vs_fp64"] = {"mean": rel(a.mean, b.mean), "var": rel(a.var, b.var), "draws_16": rel(da, db)}
    model.use_i8 = True
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--grid", type=int, default=4096)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    out = device_info()
    side = torch.linspace(-1, 1, a.grid, dtype=F64, device="cuda")
    xs = torch.stack(torch.meshgrid(side, side, indexing="ij"), -1).reshape(-1, 2).contiguous()
    g32 = torch.linspace(-1, 1, 32, dtype=F64, device="cuda")
    knots = torch.stack(torch.meshgrid(g32, g32, indexing="ij"), -1).reshape(-1, 2).contiguous()
    m316 = exact_model(316)
    out["n316"] = case(m316, None, xs, a.reps)
    out["n316_knots1024"] = case(m316, knots, xs, a.reps)
    out["n4096"] = case(exact_model(4096), None, xs, a.reps)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
