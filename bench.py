#!/usr/bin/env python3
"""Headline benchmark: SVGP-Gibbs ELBO steps/s at BASELINE.json config 2 (sparse multivariate Gibbs SVGP, synthetic 3-D
inputs, N = 2^20, M = 1024 inducing points, global minibatch 65536, fp64), rows of each minibatch sharded over the ranks.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--variant full|diag] [--impl reference] [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py ...

One step = field interpolation -> K(X_B,Z) -> Kzz Cholesky -> whitened predictive mean/variance -> Gaussian E[log-lik] +
KL -> analytic backward -> ONE NCCL all-reduce of the flat gradient -> Adam (SURVEY.md 8d).  Prints ONE JSON line.
`--impl reference` times the reference's CPU path (its pure-PyTorch restatement, oracle/, with autograd; GPyTorch is not
installable here) on the host cores, on a bounded row sample, scaled to the same metric."""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TOTAL, M_IND, B_GLOBAL, DIM = 1 << 20, 1024, 65536, 3
# dram__bytes_read.sum + dram__bytes_write.sum of one o8_rowquad_kernel launch at Bl = 65536 from the ncu --set full capture
# summarised in profiles/ (None until that capture exists for the current kernel)
TRAFFIC_ROWQUAD_BYTES = 983.2e6  # dram__bytes_read.sum + dram__bytes_write.sum of o8_rowquad_kernel at the C2 shapes, one launch:
# 477.8 + 505.4 MB (profiles/r02_ncu_full_step_kernels_final.txt)


def env_int(k, d):
    return int(os.environ.get(k, d))


# ----------------------------------------------------------------------------------------------------------------------
def make_params(variant, M, d, seed=173):
    """Initial parameters per SURVEY.md 8(d) C2 (identical on every rank: generated on CPU from one seed)."""
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    kw = dict(m=1e-3 * torch.randn(M, generator=g, dtype=f64), Ls=torch.eye(M, dtype=f64), outputscale=0.644,
              noise=0.011)
    if variant == "diag":
        kw.update(log_ell_z=math.log(0.3) + 0.1 * torch.randn(d, M, generator=g, dtype=f64),
                  prior_c=torch.full((d,), math.log(0.3), dtype=f64), prior_os=torch.ones(d, dtype=f64),
                  prior_lam=torch.full((d, d), 1.3, dtype=f64))
    else:
        Dd = torch.randn(d, generator=g, dtype=f64)
        Dd = torch.sign(Dd) * Dd.abs().clamp_min(1.2)  # 3-D Sigma(h) is PD only for |D_kk| >~ 0.6; margin for training (DESIGN.md)
        kw.update(H=torch.randn(M, d, generator=g, dtype=f64), Dm=torch.diag(Dd), row_os=1.0,
                  row_lam=torch.ones(d, dtype=f64))
    return kw


def make_data(N, d, seed=173):
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(N, d, generator=g, dtype=torch.float64) * 2 - 1
    y = torch.sin(3 * x[:, 0]) + 0.5 * torch.cos(5 * x[:, 1] * x[:, 2]) + 0.1 * torch.randn(N, generator=g,
                                                                                          dtype=torch.float64)
    perm = torch.randperm(N, generator=g)
    return x, y, perm


class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
def _inv_softplus(v: float) -> float:
    return v + math.log(-math.expm1(-v))


def oracle_step(variant, x, y, Z, kw, threads, repeats=2, chunk=2048):
    """One -ELBO forward + autograd backward of the CPU oracle (oracle/gibbs_oracle.py, the restated reference path) on the
    given rows with the bench's parameters.  Returns (best seconds, loss, gradients by parameter name).  Imports nothing
    from the product package."""
    from oracle import gibbs_oracle as o
    torch.set_num_threads(threads)
    c = lambda t: t.detach().cpu().clone()
    P = dict(Z=c(Z), m=c(kw["m"]), Ls=c(kw["Ls"]),
             raw_outputscale=c(kw["raw_outputscale"]).reshape(()) if "raw_outputscale" in kw else
             torch.tensor(_inv_softplus(kw["outputscale"]), dtype=torch.float64),
             raw_noise=c(kw["raw_noise"]).reshape(()) if "raw_noise" in kw else
             torch.tensor(_inv_softplus(kw["noise"] - 1e-4), dtype=torch.float64))
    if variant == "diag":
        P["log_ell_z"] = c(kw["log_ell_z"])
        extra = lambda: dict(log_ell_z=P["log_ell_z"], prior_c=c(kw["prior_c"]), prior_os=c(kw["prior_os"]),
                             prior_lam=c(kw["prior_lam"]))
    else:
        P["H"], P["D"] = c(kw["H"]), c(kw["Dm"])
        extra = lambda: dict(H=P["H"], Dm=P["D"], row_os=torch.tensor(float(kw["row_os"]), dtype=torch.float64),
                             row_lam=c(kw["row_lam"]))
    for v in P.values():
        v.requires_grad_(True)
    x, y = c(x), c(y)
    best, loss = float("inf"), None
    for it in range(repeats + 1):
        for v in P.values():
            v.grad = None
        t0 = time.perf_counter()
        loss = -o.svgp_gibbs_elbo(x, y, N_TOTAL, P["Z"], P["m"], P["Ls"], P["raw_outputscale"], P["raw_noise"], variant,
                                  chunk=chunk, **extra())
        loss.backward()
        dt = time.perf_counter() - t0
        if it > 0 or repeats == 0:
            best = min(best, dt)
    grads = {k: v.grad.detach().reshape(-1) if v.grad is not None else torch.zeros(v.numel(), dtype=torch.float64)
             for k, v in P.items()}
    grads["Ls"] = torch.tril(P["Ls"].grad.detach()).reshape(-1)
    return best, float(loss.detach()), grads


def headline_sample(variant, rows):
    """The bench's own inputs: first `rows` rows of minibatch 0, the same inducing points and initial parameters."""
    x_h, y_h, perm = make_data(N_TOTAL, DIM)
    return x_h[:rows].contiguous(), y_h[:rows].contiguous(), x_h[perm[:M_IND]].contiguous(), make_params(variant, M_IND, DIM)


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    threads = os.cpu_count() or 1
    rows = args.ref_rows
    x, y, Z, kw = headline_sample(args.variant, rows)
    times = []
    for i in range(args.warmup + args.steps):
        t, _, _ = oracle_step(args.variant, x, y, Z, kw, threads, repeats=0)
        if i >= args.warmup:
            times.append(t)
    t_step = sum(times) / len(times) * (B_GLOBAL / rows)
    val = 1.0 / t_step
    sample = "first %d of the %d rows of minibatch 0 per step (same x, y, Z, parameters as the GPU arm; M=%d), time scaled " \
             "x%d; fwd+autograd bwd, torch %s CPU fp64" % (rows, B_GLOBAL, M_IND, B_GLOBAL // rows, torch.__version__)
    line = {"impl": "reference", "metric": "SVGP-Gibbs ELBO steps/s", "value": val, "unit": "steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": val, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def dump_outputs(dirname, model, loss):
    """What a caller of the timed step holds after its last step, one float64 DIR/<name>.npy per array: the loss, every
    parameter after the Adam update and every gradient of that step (about 17 MB at M = 1024).  The inputs are seeded, so
    two builds run with the same arguments can be compared array for array.  The kernels accumulate with FP64 atomics and
    Adam carries the rounding differences into later steps, so even two runs of one build agree to a tolerance, not bit for
    bit (on a B200 at its 1000 W limit, after 10 + 37 steps: loss to 5e-6 relative)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    arrays = {"loss": loss.reshape(1)}
    arrays.update({"param_" + k: v for k, v in model.p.items()})
    arrays.update({"grad_" + k: v for k, v in model.g.items()})
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), t.detach().cpu().numpy())


def workload_config(args):
    return {"workload": "BASELINE config 2: sparse multivariate Gibbs SVGP, synthetic 3-D inputs, N=2^20, M=1024, "
                        "global minibatch 65536, fp64" + ("" if args.variant == "full" else " [diagonal-Gibbs variant]"),
            "kernel_variant": args.variant, "N": N_TOTAL, "M": M_IND, "global_batch": B_GLOBAL, "d": DIM,
            "parallelism": "rows of each minibatch sharded over ranks, one NCCL all-reduce of the flat gradient",
            "l2": "per-step K and T matrices are 512 MiB each (> 126 MB L2), so no explicit flush"}


# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from nonstationary_precip_b200 import ops
    from nonstationary_precip_b200._lib import check, lib, ptr, stream
    from nonstationary_precip_b200.svgp import SVGPGibbs

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus:
        if rank == 0 and world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # libraries (NCCL's version banner) write to fd 1; keep stdout clean for the single JSON line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    def allmax(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    x_h, y_h, perm = make_data(N_TOTAL, DIM)
    kw = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in make_params(args.variant, M_IND, DIM).items()}
    Z = x_h[perm[:M_IND]].to(dev)
    model = SVGPGibbs(args.variant, Z, N_TOTAL, **kw)
    model.rowquad_impl = args.gemm
    c_engine = args.engine == "c" and args.gemm == "i8" and M_IND % 128 == 0
    if c_engine:
        model.use_c_engine()
    X, Y = x_h.to(dev), y_h.to(dev)  # whole data set resident in HBM (33 MB)
    Bl = B_GLOBAL // world
    nb = N_TOTAL // B_GLOBAL
    torch_all_reduce = (lambda t: dist.all_reduce(t)) if world > 1 else None
    all_reduce = torch_all_reduce
    if c_engine and world > 1:  # the collective goes through the C ABI too (npgp_allreduce_f64 on an npgp communicator)
        from nonstationary_precip_b200.comm import NpgpComm
        all_reduce = NpgpComm(rank, world, dev)

    def rows(k):
        lo = (k % nb) * B_GLOBAL + rank * Bl
        return lo, lo + Bl

    launches_per_replay = 0
    if args.exec == "graph":
        c0 = lib().npgp_launch_count()
        # the NCCL all-reduce of the flat gradient and the Adam update are captured too: one graph launch per step and rank
        model.capture(Bl, world, B_GLOBAL, lr=args.lr, all_reduce=all_reduce, buffers=2)
        # capture() runs the step 3 times (2 warm-ups + the captured one); the captured graph holds one step's launches
        launches_per_replay = (lib().npgp_launch_count() - c0) // 4  # 2 warm-ups + one captured step per input buffer

    def train(xs, ys):
        if args.exec == "graph":
            return model.train_step_graph(xs, ys)
        return model.train_step(xs, ys, lr=args.lr, world_size=world, B_global=B_GLOBAL, all_reduce=all_reduce)

    def step_resident(k):
        lo, hi = rows(k)
        return train(X[lo:hi], Y[lo:hi])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # every phase (timed, end-to-end, profiled) restarts from the same parameters and optimiser state
    snap = model.snapshot()

    # ---- device-resident timing
    for k in range(args.warmup):
        step_resident(k)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib().npgp_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(args.steps):
        loss = step_resident(args.warmup + k)
    ev1.record()
    barrier()
    ms = allmax(ev0.elapsed_time(ev1))
    launches = lib().npgp_launch_count() - l0 + launches_per_replay * args.steps
    clocks = sampler.stop() if rank == 0 else None
    final_loss = loss.item()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, loss)

    # ---- end to end: minibatch from pinned host memory every step, loss read back every step
    xp, yp = x_h.pin_memory(), y_h.pin_memory()
    xb = torch.empty(Bl, DIM, dtype=torch.float64, device=dev)
    yb = torch.empty(Bl, dtype=torch.float64, device=dev)

    def step_e2e(k):
        lo, hi = rows(k)
        if args.exec == "graph":  # train_step_graph copies host -> static device buffers itself
            return train(xp[lo:hi], yp[lo:hi]).item()
        xb.copy_(xp[lo:hi], non_blocking=True)
        yb.copy_(yp[lo:hi], non_blocking=True)
        return train(xb, yb).item()

    model.restore(snap)
    for k in range(min(2, args.warmup)):
        step_e2e(k)
    barrier()
    t0 = time.perf_counter()
    if args.exec == "graph":
        # public pipelined API: every step still copies ITS minibatch from pinned host memory and reads ITS loss back inside
        # the timed region; the copy of step k + 1 runs under step k (second static input buffer, copy stream) and the loss of
        # step k is read while step k + 1 runs
        prev = None
        for k in range(args.steps):
            lo, hi = rows(args.warmup + k)
            ticket = model.train_step_graph_async(xp[lo:hi], yp[lo:hi])
            if prev is not None:
                model.loss_result(prev)
            prev = ticket
        model.loss_result(prev)
    else:
        for k in range(args.steps):
            step_e2e(args.warmup + k)
    barrier()
    e2e_ms = allmax((time.perf_counter() - t0) * 1e3)

    # ---- per-kernel evidence for the roofline (CUDA events around the sections of a few extra steps)
    model.restore(snap)
    model.overlap = False
    if c_engine:  # the section brackets live in the Python orchestration (same kernels, same order)
        model.engine, all_reduce_c, all_reduce = "python", all_reduce, torch_all_reduce
    for k in range(2):  # unprofiled eager steps first: the eager allocator pool (K, T: 512 MiB each) is cold after graphs
        lo, hi = rows(k)
        model.train_step(X[lo:hi], Y[lo:hi], lr=args.lr, world_size=world, B_global=B_GLOBAL, all_reduce=all_reduce)
    model.restore(snap)
    model.profile = {}
    for k in range(3):  # eager, one stream, so that the CUDA-event brackets see each section alone
        lo, hi = rows(k)
        model.overlap = False
        model.train_step(X[lo:hi], Y[lo:hi], lr=args.lr, world_size=world, B_global=B_GLOBAL, all_reduce=all_reduce)
        model.overlap = True
    torch.cuda.synchronize()
    sec = model.section_ms()
    model.profile = None
    if c_engine:
        model.engine, all_reduce = "c", all_reduce_c
    out = torch.zeros(8, dtype=torch.float64, device=dev)
    peak_tf = 0.0
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        check(lib().npgp_fp64_peak_probe(1, 148 * 8, 2048, ptr(out), stream()), "probe")
        b.record()
        b.synchronize()
        peak_tf = max(peak_tf, 148 * 8 * 2048 * 8 * 16 * 512 / a.elapsed_time(b) / 1e9)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    rq_tf = 2.0 * Bl * M_IND * M_IND / sec["rowquad"] / 1e9
    i8_roof = None
    if args.gemm == "i8":
        # dominant kernel of the int8 path: o8_rowquad_kernel, timed alone on the digit planes the last step left in the
        # model's buffers (real data), average of 5 launches with CUDA events on the launching stream
        from nonstationary_precip_b200 import ops as _ops
        wb = model._digit_buffers(Bl)
        s_dev = torch.nn.functional.softplus(model.p["raw_outputscale"])
        gvec = torch.randn(Bl, dtype=torch.float64, device=dev)
        times = []
        for it in range(7):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _ops.o8_rowquad_digits(Bl, M_IND, wb["Ad"], s_dev, wb["Cd"], wb["cexp"], wb["T"], q_part=wb["q_part"], gvec=gvec,
                                   du_part=wb["du_part"])
            b.record()
            b.synchronize()
            if it >= 2:
                times.append(a.elapsed_time(b))
        rq_ms = sum(times) / len(times)
        top = 28 * 2.0 * Bl * M_IND * M_IND / rq_ms / 1e9  # 28 int8 digit products per FP64-exact product

        def i8_probe(n_tile, coll, reps=4096):
            best = float("inf")
            for _ in range(3):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                check(lib().npgp_i8_peak_probe(n_tile, coll, 148, reps, stream()), "i8 probe")
                b.record()
                b.synchronize()
                best = min(best, a.elapsed_time(b))
            return 148.0 * reps * 8 * 2 * 128 * n_tile * 32 / best / 1e9  # TOP/s

        i8_peak = i8_probe(256, 0)
        i8_roof = {"bound": "tensor", "kernel": "o8_rowquad_kernel (T = K C as 28 exact int8 byte-digit products, tcgen05 "
                                                "kind::i8 + TMEM; row dot and K^T g fused)", "achieved": top, "peak": i8_peak,
                   "unit": "TFLOP/s", "frac": top / i8_peak, "ms": rq_ms,
                   "fp64_equivalent_tflops": 2.0 * Bl * M_IND * M_IND / rq_ms / 1e9,
                   # algorithmic bytes per launch: A digit planes read once (7 B/entry) + T written (8 B/entry) + C planes
                   "algorithmic_bytes": (7.0 + 8.0) * Bl * M_IND + 7.0 * M_IND * M_IND,
                   "traffic": TRAFFIC_ROWQUAD_BYTES if (world == 1 and TRAFFIC_ROWQUAD_BYTES) else None,
                   "peak_source": "measured in this run: npgp_i8_peak_probe, back-to-back tcgen05.mma kind::i8 128x256x32 from "
                                  "resident shared memory on 148 SMs (MEASURED_PEAKS.json has no int8 entry; 2 x its bf16 "
                                  "burst figure would be %.0f); unit is int8 TOP/s" % (2.0 * peaks.get("bf16_tflops", 0.0)),
                   "tile_shape_ceiling": {"what": "same probe at the engine's 128x64x32 tile shape (TMEM holds 7 accumulators "
                                                  "of 64 columns): shared-memory operand feed bound",
                                          "plain": i8_probe(64, 0), "collector_a_reuse": i8_probe(64, 1)}}
    kxz_gbs = 16.0 * Bl * M_IND / (sec["kxz_fwd"] + sec["kxz_bwd"]) / 1e6

    # ---- parity at the headline size, in the same run: the GPU path and the CPU oracle on the SAME rows (the first
    # ref_rows rows of minibatch 0), the same Z and the same parameters; the oracle pass is also the CPU baseline timing
    parity = t_cpu = None
    if rank == 0 and world == 1:
        threads = os.cpu_count() or 1
        cpu_rows = args.ref_rows
        model.restore(snap)
        for k in range(3):  # a few optimiser steps first: at the initial S = I the quadratic term T = K C is identically 0
            step_resident(k)
        state = dict(kw, **{k: v.detach().clone() for k, v in model.p.items()})
        state["Dm"] = state.get("D")
        got_loss = float(model.loss_and_grad(X[:cpu_rows], Y[:cpu_rows], 1, cpu_rows))
        info = int(model.last["info"])
        got = {k: v.detach().reshape(-1).cpu().clone() for k, v in model.g.items()}
        sec_cpu, want_loss, want = oracle_step(args.variant, x_h[:cpu_rows], y_h[:cpu_rows], state["Z"], state, threads)
        t_cpu = sec_cpu * (B_GLOBAL / cpu_rows)
        grel = {k: float((got[k] - want[k]).abs().max() / want[k].abs().max().clamp_min(1e-300)) for k in want}
        parity = {"elbo_rel": abs(got_loss - want_loss) / abs(want_loss), "grad_rel_max": max(grel.values()),
                  "grad_rel": grel, "rows": cpu_rows, "M": M_IND, "tol": 1e-6, "cholesky_info": info,
                  "state": "parameters after 3 Adam steps from the bench's initial state",
                  "against": "oracle/gibbs_oracle.py svgp_gibbs_elbo + autograd on the same x, y, Z and parameters"}
        parity["ok"] = bool(parity["elbo_rel"] <= 1e-6 and parity["grad_rel_max"] <= 1e-6 and info == 0)

    line = None
    if rank == 0:
        threads = os.cpu_count() or 1
        cpu_rows = args.ref_rows
        line = {
            "metric": "SVGP-Gibbs ELBO steps/s", "value": args.steps / (ms / 1e3), "unit": "steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64",
            "data": "synthetic",
            "config": workload_config(args),  # identical in both arms
            "impl_detail": {"engine": "npgp_svgp_step: one C-ABI call per step (forward, analytic backward, all-reduce, guarded "
                                      "Adam)" if c_engine else "python orchestration of the C-ABI kernels (svgp.py)",
                            "exec": "cuda_graph + 3 streams" if args.exec == "graph" else "eager",
                            "gemm": "FP64 DMMA" if args.gemm == "dmma" else
                            "FP64-exact int8 byte-digit products on tcgen05 (28 per product, int32 accumulation); "
                                    "K(X,Z) stored as 7-byte digits only"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": args.steps / (e2e_ms / 1e3), "unit": "steps/s",
                    "h2d_bytes_per_step": Bl * (DIM + 1) * 8 * world, "d2h_bytes_per_step": 8 * world},
            "roofline": i8_roof if i8_roof is not None else {
                         "bound": "tensor", "kernel": "dgemm_kernel (rowquad T = K C, FP64 DMMA)", "achieved": rq_tf,
                         "peak": peak_tf, "unit": "TFLOP/s", "frac": rq_tf / peak_tf,
                         # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at Bl = 65536 from the ncu --set full
                         # capture in profiles/r01_ncu_rowquad_full_summary.txt (algorithmic: 1082 MB)
                         "traffic": 1.0542e9 if world == 1 else None,
                         "peak_source": "in-run DMMA.8x8x4 probe; MEASURED_PEAKS.json has no FP64 entry "
                                        "(nominal 148 SM x 64 FMA x 2 x 1.965 GHz = 37.2)"},
            "roofline_kxz": {"bound": "hbm", "kernel": "gibbs_%s fwd+bwd (K written, T read: 16 B/pair)" % args.variant,
                             "achieved": kxz_gbs, "peak": hbm, "unit": "GB/s", "frac": kxz_gbs / hbm,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650",
                             # the roof these tile kernels actually sit under: FP64 instructions per pair counted in the SASS of
                             # the inner loops (cuobjdump, DESIGN.md section 4) x pairs / measured time, against the DFMA issue
                             # peak of 148 SMs x 64 lanes x 1.965 GHz; ncu: sm__pipe_fp64_cycles_active 75 % (fwd) / 65 % (bwd)
                             "fp64_pipe": None if args.variant != "full" else {
                                 "dp_instr_per_pair": {"fwd": 73, "bwd": 160},
                                 "achieved_dp_instr_per_s": (73 + 160) * float(Bl) * M_IND / ((sec["kxz_fwd"] + sec["kxz_bwd"]) * 1e-3),
                                 "peak_dp_instr_per_s": 148 * 64 * 1.965e9,
                                 "frac": (73 + 160) * float(Bl) * M_IND / ((sec["kxz_fwd"] + sec["kxz_bwd"]) * 1e-3) / (148 * 64 * 1.965e9),
                                 "ncu_pipe_fp64_active": {"fwd": 0.751, "bwd": 0.647,
                                                          "source": "profiles/r02_ncu_full_step_kernels_final.txt"}}},
            # one eager single-stream step, CUDA events per section (sections overlap in the timed graph replay):
            # replicated = work every rank repeats (O(M^3) chain on Kzz, assembly, all-reduce, Adam); sharded = work on this
            # rank's B/G rows.  The Amdahl table in DESIGN.md is built from these.
            "sections_ms": {k: round(v, 4) for k, v in sec.items()},
            "sections_split_ms": {
                "replicated": round(sum(v for k, v in sec.items() if k.startswith(("zz_fwd", "m3_bwd", "assemble", "allreduce",
                                                                                  "adam"))), 4),
                "sharded": round(sum(v for k, v in sec.items() if not k.startswith(("zz_fwd", "m3_bwd", "assemble", "allreduce",
                                                                                    "adam"))), 4)},
            "final_loss": final_loss,
        }
        if t_cpu is not None:
            line["cpu_baseline"] = {
                "value": 1.0 / t_cpu, "unit": "steps/s", "cores": threads, "kind": "port",
                "sample": "first %d of the %d rows of minibatch 0 (same x, y, Z, parameters as the GPU arm; M=%d) fwd+autograd "
                          "bwd of the oracle, time scaled x%d" % (cpu_rows, B_GLOBAL, M_IND, B_GLOBAL // cpu_rows)}
            line["parity"] = parity

    # ---- the other shardable paths (prediction, DSVI, streamed SGPR): short legs with their own parity, under "configs".
    # A watchdog prints the headline line without them if a leg stalls, so they can never cost the headline number.
    emitted = threading.Event()

    def emit(configs):
        if emitted.is_set():
            return
        emitted.set()
        if rank == 0:
            line["configs"] = configs
            sys.stdout.flush()
            os.dup2(real_stdout, 1)
            print(json.dumps(line), flush=True)
            os.dup2(2, 1)

    legs = [s for s in args.legs.split(",") if s and s != "none"]
    rc = 3 if (parity is not None and not parity["ok"]) else 0  # a fast step whose results differ from the reference's is not a result
    if legs:
        def on_timeout():
            emit({"error": "legs exceeded %d s; headline line printed without them" % args.legs_timeout})
            sys.stdout.flush()
            os._exit(rc)

        dog = threading.Timer(args.legs_timeout, on_timeout)
        dog.daemon = True
        dog.start()
        model._graph = None  # free the step graph's memory pool first
        model._i8_bufs.clear()
        torch.cuda.empty_cache()
        import bench_legs
        configs = bench_legs.run_all(rank, world, dev, allmax, all_reduce, make_params, which=legs)
        dog.cancel()
        emit(configs)
        if any(isinstance(v, dict) and isinstance(v.get("parity"), dict) and not v["parity"].get("ok", True) for v in configs.values()):
            rc = rc or 4
    else:
        emit({})
    if world > 1:
        # The captured step graph holds NCCL kernels; tearing the communicator down while that graph is alive hung
        # (measured: the line was printed, then destroy_process_group never returned).  Drop the graph, drain the device,
        # meet the other ranks once more and leave without the NCCL teardown.
        model._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(rc)
    if rc:
        sys.exit(rc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", default="full", choices=["full", "diag"])
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--gemm", default="i8", choices=["dmma", "i8"],
                    help="row-quadratic GEMM: FP64 DMMA (dgemm.cu) or exact int8 Ozaki split on tcgen05 (ozaki.cu)")
    ap.add_argument("--engine", default="c", choices=["c", "python"],
                    help="c: the whole step is one C-ABI call (npgp_svgp_step); python: kernel-by-kernel orchestration in svgp.py")
    ap.add_argument("--exec", default="graph", choices=["graph", "eager"],
                    help="replay the step as a captured CUDA graph (default) or launch it eagerly")
    ap.add_argument("--ref-rows", type=int, default=16384, help="minibatch rows the CPU reference processes per step")
    ap.add_argument("--legs", default="c5,c4,c3", help="extra legs reported under \"configs\" (comma list of c5,c4,c3; none)")
    ap.add_argument("--legs-timeout", type=int, default=240, help="seconds after which the legs are abandoned")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss, parameters and gradients of the last one to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU step computed; --impl reference has no such step")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
