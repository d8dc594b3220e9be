#!/usr/bin/env python3
"""BASELINE config 1 end to end on the B200 kernels: MAP training of the diagonal-Gibbs GP on the Upper-Indus-Basin
precipitation table (394 rows: lon, lat, tp), 80/20 random splits, RMSE / NLPD on the held-out rows.

Same experiment as the reference's experiments/spatial_exp.py:97-231 (data preparation :113-141, prior set-up :155-166,
model / hyper-parameter freezing :170-187, Adam loop :192-210, evaluation :214-231) with the same option names and
defaults (:54-81).  Differences, all forced by defects of that script (SURVEY Appendix D): the test predictive is taken
from `model.predict` (the script's eval-mode `model(x_test)` feeds n-row lengthscales to an (n + n*)-row kernel), the
plotting tail (cartopy, a results CSV that is not in the repository) is dropped, and the inducing points of the sparse
variant come from `utils.dataprep.kmeans_inducing_points` instead of pymc3.

    python experiments/spatial_exp.py --n_iter 5000 --splits 10 [--inference sparse --M 250] [--data path/to.csv]
        [--map_grid 1000 --map_samples 16 --map_out map.npz]

With --map_grid G the model of the last split also predicts over a G x G grid of the data's bounding box through its
posterior() snapshot (write_map), at any G the device memory allows.

Without --data the table is read from tests/golden/uib_spatial_dataprep.npz (the reference's data fixture, exported by
tests/golden/make_golden.py).  Needs a GPU: the models run on the npgp CUDA kernels only."""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from nonstationary_precip_b200.gp_base import ExactMarginalLogLikelihood, GaussianLikelihood  # noqa: E402
from nonstationary_precip_b200.models.gibbs_kernels import LogNormalPriorProcess  # noqa: E402
from nonstationary_precip_b200.models.nonstationary_models import DiagonalExactGP, DiagonalSparseGP  # noqa: E402
from nonstationary_precip_b200.utils.config import BASE_SEED  # noqa: E402
from nonstationary_precip_b200.utils.dataprep import kmeans_inducing_points  # noqa: E402
from nonstationary_precip_b200.utils.metrics import get_trainable_param_names, nlpd, rmse  # noqa: E402


def load_khyber_data(path=None):
    """(x (n,2) lon/lat, y (n,) precipitation) in float64, as experiments/spatial_exp.py:36-40."""
    if path is None:
        raw = np.load(os.path.join(ROOT, "tests", "golden", "uib_spatial_dataprep.npz"))["raw"]
    else:
        import pandas as pd
        raw = np.asarray(pd.read_csv(path, dtype=np.float64))
    return torch.tensor(raw[:, 0:2], dtype=torch.float64), torch.tensor(raw[:, -1], dtype=torch.float64)


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--data", default=None)
    p.add_argument("--inference", default="exact", choices=["exact", "sparse"])
    p.add_argument("--train_percent", type=float, default=80.0)
    p.add_argument("--lr", type=float, default=1e-2)
    p.add_argument("--n_iter", type=int, default=5000)
    p.add_argument("--splits", type=int, default=10)
    p.add_argument("--M", type=int, default=250)
    p.add_argument("--prior_scale", type=float, default=1.0)
    p.add_argument("--prior_ell", type=float, default=1.3)
    p.add_argument("--prior_mean", type=float, default=0.3)
    p.add_argument("--noise", type=float, default=0.011, help="0: learn the noise, else fixed")
    p.add_argument("--scale", type=float, default=0.644, help="0: learn the outputscale, else fixed")
    p.add_argument("--log_every", type=int, default=400)
    p.add_argument("--json", default=None, help="write the per-split metrics here")
    p.add_argument("--map_grid", type=int, default=0,
                   help="G > 0: after the last split, predict over a G x G grid spanning the data's bounding box")
    p.add_argument("--map_samples", type=int, default=0, help="posterior sample fields drawn over the map grid")
    p.add_argument("--map_out", default="spatial_map.npz", help="where the map arrays are written (.npz)")
    return p.parse_args(argv)


def make_prior(args, device):
    prior = LogNormalPriorProcess(input_dim=2).to(device).double()
    prior.covar_module.outputscale = args.prior_scale * torch.ones_like(prior.covar_module.outputscale)
    prior.covar_module.base_kernel.lengthscale = args.prior_ell * torch.ones_like(
        prior.covar_module.base_kernel.lengthscale)
    prior.mean_module.constant = torch.nn.Parameter(
        math.log(args.prior_mean) * torch.ones_like(prior.mean_module.constant))
    for p in prior.parameters():
        p.requires_grad = False
    return prior


def run_split(i, x, y, args, device, log=print):
    rng = np.random.default_rng(BASE_SEED + i)
    torch.manual_seed(BASE_SEED + i)
    stdx, meanx = torch.std_mean(x, dim=-2)
    stdy, meany = torch.std_mean(y)
    x_norm, y_norm = (x - meanx) / stdx, (y - meany) / stdy
    num_train = math.ceil(args.train_percent / 100 * y.shape[0])
    idx = np.arange(0, y.shape[0], 1)
    rng.shuffle(idx)
    tr, te = idx[:num_train], idx[num_train:]
    x_train, y_train = x_norm[tr].to(device).contiguous(), y_norm[tr].to(device).contiguous()
    x_test, y_test = x_norm[te].to(device).contiguous(), y_norm[te].to(device).contiguous()

    prior = make_prior(args, device)
    likelihood = GaussianLikelihood().to(device).double()
    if args.inference == "exact":
        model = DiagonalExactGP(x_train, y_train, likelihood, prior, num_dim=2).to(device).double()
    else:
        z = kmeans_inducing_points(min(args.M, num_train), x_train, seed=BASE_SEED + i)
        model = DiagonalSparseGP(x_train, y_train, likelihood, prior, z, num_dim=2).to(device).double()
    if args.noise > 0:
        model.likelihood.noise = args.noise
        for p in model.likelihood.noise_covar.parameters():
            p.requires_grad = False
    if args.scale > 0:
        model.covar_module.outputscale = args.scale
        model.covar_module._parameters["raw_outputscale"].requires_grad = False
    model.train()
    likelihood.train()
    optimizer = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=args.lr)
    mll = ExactMarginalLogLikelihood(likelihood, model)
    losses = []
    t0 = time.perf_counter()
    for it in range(args.n_iter):
        optimizer.zero_grad()
        loss = -mll(model(x_train), y_train)
        loss.backward()
        if it % args.log_every == 0 or it == args.n_iter - 1:
            losses.append(loss.item())
            log("Iter %d/%d - Loss: %.3f  amplitude: %.3f noise: %.3f" % (
                it + 1, args.n_iter, losses[-1], model.covar_module.outputscale.item(), model.likelihood.noise.item()))
        optimizer.step()
    torch.cuda.synchronize()
    train_s = time.perf_counter() - t0

    model.eval()
    likelihood.eval()
    with torch.no_grad():
        pred_y_test = likelihood(model.predict(x_test))
    rmse_test = float(rmse(pred_y_test.loc.detach(), y_test, stdy))
    nlpd_test = float(nlpd(pred_y_test, y_test, stdy.to(device)))
    if args.map_grid > 0 and i == args.splits - 1:
        write_map(model, x_norm, meanx, stdx, meany, stdy, args)
    return dict(split=i, rmse=rmse_test, nlpd=nlpd_test, first_loss=losses[0], last_loss=losses[-1],
                train_s=train_s, steps_per_s=args.n_iter / train_s, trainable=get_trainable_param_names(model))


def write_map(model, x_norm, meanx, stdx, meany, stdy, args):
    """Posterior over a G x G grid spanning the bounding box of the normalised inputs, streamed through the model's
    posterior() snapshot: mean and var_y in the original units of the target, the lengthscale field (D, G, G) in normalised
    input units and `map_samples` correlated draws of f in the target's units.  Row i of a (G, G) map is latitude i, column
    j longitude j; lon / lat (G,) are the grid axes in the original units."""
    G = args.map_grid
    lo, hi = x_norm.min(0).values, x_norm.max(0).values
    axes = [torch.linspace(float(lo[d]), float(hi[d]), G, dtype=torch.float64) for d in range(2)]
    lat, lon = torch.meshgrid(axes[1], axes[0], indexing="ij")
    xs = torch.stack([lon.reshape(-1), lat.reshape(-1)], 1).to(model.train_inputs[0].device)
    post = model.posterior()
    pred = post.predictive(xs, field=True)
    out = dict(lon=(axes[0] * stdx[0] + meanx[0]).numpy(), lat=(axes[1] * stdx[1] + meanx[1]).numpy(),
               mean=(pred.mean * stdy + meany).reshape(G, G).cpu().numpy(),
               var_y=(pred.var_y * stdy ** 2).reshape(G, G).cpu().numpy(),
               ell=pred.field.reshape(-1, G, G).cpu().numpy())
    if args.map_samples > 0:
        draws = post.sample(xs, args.map_samples, seed=BASE_SEED)
        out["samples"] = (draws * stdy + meany).reshape(-1, G, G).cpu().numpy()
    np.savez(args.map_out, **out)
    print("Map %d x %d (%d draws) written to %s" % (G, G, args.map_samples, args.map_out))


def main(argv=None):
    args = parse_args(argv)
    if not torch.cuda.is_available():
        raise RuntimeError("experiments/spatial_exp.py needs a CUDA device (the models have no CPU path)")
    device = torch.device("cuda")
    x, y = load_khyber_data(args.data)
    results = []
    for i in range(args.splits):
        print("Running split " + str(i))
        r = run_split(i, x, y, args, device)
        print("RMSE test =  %.4f\nNLPD test = %.4f" % (r["rmse"], r["nlpd"]))
        results.append(r)
    rm, nl = np.array([r["rmse"] for r in results]), np.array([r["nlpd"] for r in results])
    k = math.sqrt(len(results))
    print("Final RMSE across splits: %.4f +- %.4f" % (rm.mean(), rm.std() / k))
    print("Final NLPD across splits: %.4f +- %.4f" % (nl.mean(), nl.std() / k))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(args=vars(args), splits=results, rmse_mean=rm.mean(), nlpd_mean=nl.mean()), f, indent=1)
    return results


if __name__ == "__main__":
    main()
