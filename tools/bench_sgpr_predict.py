#!/usr/bin/env python3
"""Streamed SGPR prediction at scale: posterior() and posterior().predictive() of both SGPR models (sgpr.py).  Prints ONE
JSON line with the device name and power limit read in the same run.

  python tools/bench_sgpr_predict.py [--reps 3] [--grid 4096] [--train 1048576] [--st-rows 1048576]

  (a) diagonal model (SGPRGibbsStream), M = 1024, d = 2: posterior() over `train` rows, then predictive rows/s on the c5
      grid (grid x grid rows on [-1, 1]^2, 65536-row chunks), `reps` times
  (b) spatio-temporal model (SGPRSpatioTemporalStream), M = 2048 (feature width 4096): posterior() over `train` c3-shaped
      rows (time, lon, lat), predictive rows/s on `st-rows` such rows
  (c) the row-side contraction of (a) alone, alternated in one run: the two triangular row-norm passes
      (npgp_o8_trinorm_digits against P and V) and the composition they replace, two q-only row-quadratic passes
      (npgp_o8_rowquad_digits, T = NULL) against P^T P and V^T V, on the same 65536-row planes; CUDA events over 20 launches
  (d) parity of the digit path with the FP64 path (use_i8 = False) on 4096 sampled grid rows: the dense oracle cannot hold
      the (train + test) x M root at this scale, and the FP64 path is checked against it in tests/test_sgpr_predict_gpu.py"""
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
from bench_predict import device_info, rel, timed  # noqa: E402

F64 = torch.float64
CHUNK = 65536


def diag_model(n_train, M=1024):
    from nonstationary_precip_b200.sgpr import SGPRGibbsStream
    g = torch.Generator().manual_seed(1)
    x = torch.rand(n_train, 2, generator=g, dtype=F64) * 2 - 1
    y = torch.sin(3 * x[:, 0]) * torch.cos(2 * x[:, 1]) + 0.1 * torch.randn(n_train, generator=g, dtype=F64)
    Z = x[torch.randperm(n_train, generator=g)[:M]].clone()
    le = math.log(0.2) + 0.1 * torch.randn(2, M, generator=g, dtype=F64)
    c, os_, lam = torch.full((2,), math.log(0.2), dtype=F64), torch.ones(2, dtype=F64), torch.full((2, 2), 1.3, dtype=F64)
    model = SGPRGibbsStream(Z.cuda(), le.cuda(), c.cuda(), os_.cuda(), lam.cuda(), outputscale=0.8, noise=0.05)
    return model, x.cuda(), y.cuda()


def st_rows(n, g):
    return torch.cat([torch.rand(n, 1, generator=g, dtype=F64) * 6 - 3, torch.rand(n, 2, generator=g, dtype=F64) * 2 - 1], 1)


def st_model(n_train, M=2048):
    from nonstationary_precip_b200.sgpr import SGPRSpatioTemporalStream
    g = torch.Generator().manual_seed(2)
    x = st_rows(n_train, g)
    y = torch.sin(2 * math.pi * x[:, 0] / 1.7) * torch.exp(-(x[:, 1:] ** 2).sum(-1)) + 0.1 * torch.randn(n_train, generator=g,
                                                                                                          dtype=F64)
    Z = x[torch.randperm(n_train, generator=g)[:M]].clone()
    le = math.log(0.3) + 0.1 * torch.randn(2, M, generator=g, dtype=F64)
    c, os_, lam = torch.full((2,), math.log(0.3), dtype=F64), torch.ones(2, dtype=F64), torch.full((2, 2), 1.3, dtype=F64)
    model = SGPRSpatioTemporalStream(Z.cuda(), le.cuda(), c.cuda(), os_.cuda(), lam.cuda(), hyp_t=(0.05, 0.8, 1.7, 7.6),
                                     outputscale_s=0.8, noise=0.05)
    return model, x.cuda(), y.cuda()


def bench_model(name, model, x, y, xs, reps, chunk_train):
    t_post, post = timed(lambda: model.posterior(x, y, chunk=chunk_train))
    post.predictive(xs[:CHUNK + 1000], chunk=CHUNK)  # warm-up: both chunk shapes
    ms = []
    for _ in range(reps):
        t, pred = timed(lambda: post.predictive(xs, chunk=CHUNK))
        ms.append(t)
    n = xs.shape[0]
    return post, {"what": name, "train_rows": x.shape[0], "M": model.Z.shape[0], "width": post.width, "digits": post.digits,
                  "posterior_ms": round(t_post, 1), "rows": n, "rows_per_s": [round(n / t * 1e3) for t in ms],
                  "spread": round((max(ms) - min(ms)) / min(ms), 4),
                  "finite": bool(torch.isfinite(pred.mean).all() and torch.isfinite(pred.var).all()),
                  "var_min": pred.var.min().item()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--grid", type=int, default=4096)
    ap.add_argument("--train", type=int, default=1 << 20)
    ap.add_argument("--st-rows", type=int, default=1 << 20)
    a = ap.parse_args()
    from nonstationary_precip_b200 import ops
    torch.cuda.set_device(0)
    out = device_info()

    # (a) diagonal model on the c5 grid
    model, x, y = diag_model(a.train)
    side = torch.linspace(-1, 1, a.grid, dtype=F64, device="cuda")
    xs = torch.stack(torch.meshgrid(side, side, indexing="ij"), -1).reshape(-1, 2).contiguous()
    post, out["diag_c5"] = bench_model("diag, c5 grid", model, x, y, xs, a.reps, 65536)

    # (c) triangular norms against two q-only passes, alternated
    M = post.M
    xc = xs[:CHUNK]
    ell = ops.rbf_matvec_fwd(xc, post.Z, post.prior_lam, post.prior_os, post.alpha.unsqueeze(-1), bias=post.prior_c,
                             apply_exp=True).squeeze(-1)
    Ad = torch.empty(ops.digits_bytes(CHUNK, M, 128), dtype=torch.uint8, device="cuda")
    ops.gibbs_diag_fwd_digits(xc, ell, post.Z, post.ell_z, post.one, Ad)
    _, _, (_, _, P), _ = model._z_side()
    (Pd, Pe), (Vd, Ve) = post.planes
    Pm = P.detach().contiguous()
    # the q-only baseline needs P^T P and V^T V: rebuild V = sqrt(s) P_B P as posterior() forms it
    s = torch.nn.functional.softplus(model.raw_outputscale.detach()).reshape(())
    noise = (1e-4 + torch.nn.functional.softplus(model.raw_noise.detach())).reshape(())
    from nonstationary_precip_b200 import functional as Fn
    W, _, _, _, _ = model._pass1(x, y, 65536, post.ell_z, post.alpha, Pm, None)
    _, PB = Fn.psd_safe_chol_inv(torch.eye(M, dtype=F64, device="cuda") + (s / noise) * 0.5 * (W + W.T))
    V = torch.sqrt(s) * (PB @ Pm)
    grams = []
    for X in (Pm, V):
        G = (X.T @ X).contiguous()
        d = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device="cuda")
        e = torch.empty(M, dtype=torch.int32, device="cuda")
        ops.o8_slice_rows(G, 64, d, e)
        grams.append((d, e))
    q_tri = torch.empty(2, M // 64, CHUNK, dtype=F64, device="cuda")
    q_rq = torch.empty_like(q_tri)

    def tri():
        ops.o8_trinorm_digits(CHUNK, M, M, Ad, post.one, Pd, Pe, q_tri[0])
        ops.o8_trinorm_digits(CHUNK, M, M, Ad, post.one, Vd, Ve, q_tri[1])

    def two_qonly():
        for k, (d, e) in enumerate(grams):
            ops.o8_rowquad_digits(CHUNK, M, Ad, post.one, d, e, None, q_part=q_rq[k])

    def launches(fn, reps=20):
        fn()
        t, _ = timed(lambda: [fn() for _ in range(reps)])
        return t / reps

    per = {"trinorm_P_and_V": [], "two_qonly_passes": []}
    for _ in range(3):
        per["trinorm_P_and_V"].append(round(launches(tri), 4))
        per["two_qonly_passes"].append(round(launches(two_qonly), 4))
    out["contraction_65536x1024_ms"] = per
    out["contraction_agreement"] = {"P": rel(q_tri[0].sum(0), q_rq[0].sum(0)), "V": rel(q_tri[1].sum(0), q_rq[1].sum(0))}

    # (d) digit path against the FP64 path on 4096 sampled grid rows
    idx = torch.randperm(xs.shape[0], generator=torch.Generator().manual_seed(3))[:4096].cuda()
    ref = model
    ref.use_i8 = False
    p64 = ref.posterior(x, y, chunk=65536).predictive(xs[idx])
    ref.use_i8 = True
    pdg = post.predictive(xs[idx])
    out["fp64_path_parity_4096"] = {"mean": rel(pdg.mean, p64.mean), "var": rel(pdg.var, p64.var)}
    del model, post, x, y, xs, Ad, grams, p64, pdg
    torch.cuda.empty_cache()

    # (b) spatio-temporal model, c3-shaped rows
    model, x, y = st_model(a.train)
    xs = st_rows(a.st_rows, torch.Generator().manual_seed(4)).cuda()
    _, out["st_c3"] = bench_model("spatio-temporal, c3 rows", model, x, y, xs, a.reps, 32768)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
