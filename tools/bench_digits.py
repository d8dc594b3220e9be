#!/usr/bin/env python3
"""Timings of the digit-plane path at the C2 shapes (B=65536, M=1024, d=3): Gibbs kernels emitting digits, the int8
row-quadratic kernel and the MN-major SYRK, the int8 peak probes.
Run on the GPU box:  python tools/bench_digits.py > gpurun_out/bench_digits.jsonl"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nonstationary_precip_b200 import ops  # noqa: E402
from nonstationary_precip_b200._lib import check, lib, stream  # noqa: E402


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def report(name, ms, best, **kw):
    print(json.dumps(dict(kernel=name, ms_median=round(ms, 4), ms_best=round(best, 4), **kw)), flush=True)


def main():
    torch.manual_seed(0)
    B, M, d = int(os.environ.get("B", 65536)), int(os.environ.get("M", 1024)), 3
    f64 = dict(dtype=torch.float64, device="cuda")
    x = torch.rand(B, d, **f64) * 2 - 1
    z = torch.rand(M, d, **f64) * 2 - 1
    ell_x = torch.exp(0.1 * torch.randn(d, B, **f64)) * 0.3
    ell_z = torch.exp(0.1 * torch.randn(d, M, **f64)) * 0.3
    Dm = torch.diag(torch.tensor([1.2, -1.3, 1.25], **f64))
    Sx, Sz = ops.sigma_from_h_fwd(torch.randn(B, d, **f64), Dm), ops.sigma_from_h_fwd(torch.randn(M, d, **f64), Dm)
    s = torch.tensor([0.644], **f64)
    u = torch.randn(M, **f64)
    K = torch.empty(B, M, **f64)
    digits = torch.empty(ops.digits_bytes(B, M, 128), dtype=torch.uint8, device="cuda")
    parts = torch.empty(ops.gibbs_digits_splits(B, M), B, **f64)
    pairs = B * M
    for name, fn, byt in (
            ("gibbs_full_fwd (FP64 K, 8 B/pair)", lambda: ops.gibbs_full_fwd(x, Sx, z, Sz, 1e-5, s, u=u, out=K), 8),
            ("gibbs_full_fwd_digits (7 B/pair)", lambda: ops.gibbs_full_fwd_digits(x, Sx, z, Sz, 1e-5, s, digits, u=u, Ku_part=parts), 7),
            ("gibbs_diag_fwd (FP64 K)", lambda: ops.gibbs_diag_fwd(x, ell_x, z, ell_z, s, u=u, out=K), 8),
            ("gibbs_diag_fwd_digits", lambda: ops.gibbs_diag_fwd_digits(x, ell_x, z, ell_z, s, digits, u=u, Ku_part=parts), 7)):
        ms, best = timeit(fn)
        report(name, ms, best, gbs=round(byt * pairs / best / 1e6, 1), mpairs_per_s=round(pairs / best / 1e3, 1))
    ops.gibbs_full_fwd_digits(x, Sx, z, Sz, 1e-5, s, digits, u=u, Ku_part=parts)
    A = torch.randn(M, M, **f64)
    C = A @ A.T / M - 0.3 * torch.eye(M, **f64)
    C = 0.5 * (C + C.T)
    Cd = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device="cuda")
    cexp = torch.empty(M, dtype=torch.int32, device="cuda")
    ms, best = timeit(lambda: ops.o8_slice_rows(C, 64, Cd, cexp))
    report("o8_slice_rows(C)", ms, best)
    T = torch.empty(B, M, **f64)
    q_part = torch.empty(M // 64, B, **f64)
    du_part = torch.empty((B + 127) // 128, M, **f64)
    gvec = torch.randn(B, **f64)
    part = torch.empty(max(1, ops.o8_syrk_part_bytes(B, M) // 8), **f64)
    Out = torch.empty(M, M, **f64)
    ms, best = timeit(lambda: ops.o8_rowquad_digits(B, M, digits, s, Cd, cexp, T, q_part=q_part, gvec=gvec, du_part=du_part))
    report("o8_rowquad_digits (T, q, K^T g)", ms, best, int8_tops=round(28 * 2 * B * M * M / best / 1e9, 1),
           fp64_equiv_tflops=round(2 * B * M * M / best / 1e9, 2))
    ms, best = timeit(lambda: ops.o8_rowquad_digits(B, M, digits, s, Cd, cexp, T))
    report("o8_rowquad_digits (T only)", ms, best, int8_tops=round(28 * 2 * B * M * M / best / 1e9, 1))
    ms, best = timeit(lambda: ops.o8_syrk_digits(B, M, digits, s, part, out=Out))
    report("o8_syrk_digits (MN-major planes, finish included)", ms, best,
           int8_tops_useful=round(28 * B * M * (M + 64) / best / 1e9, 1))
    Kf = ops.gibbs_full_fwd(x, Sx, z, Sz, 1e-5, s)
    ms, best = timeit(lambda: ops.rowquad_i8(Kf, C, T=T))
    report("rowquad_i8 (general operands: slicing passes included)", ms, best)
    ms, best = timeit(lambda: ops.syrk_i8(Kf, out=Out))
    report("syrk_i8 (general operands: column maxima + transposed slicing included)", ms, best)
    ms, best = timeit(lambda: ops.rowquad(Kf, C, T=T), iters=5)
    report("rowquad (FP64 DMMA)", ms, best, tflops=round(2 * B * M * M / best / 1e9, 2))
    for n_tile, coll in ((256, 0), (256, 1), (64, 0), (64, 1)):
        reps = 4096
        ms, best = timeit(lambda: check(lib().npgp_i8_peak_probe(n_tile, coll, 148, reps, stream()), "probe"), iters=5)
        report("i8_peak_probe[128x%dx32, collector=%d]" % (n_tile, coll), ms, best,
               int8_tops=round(148.0 * reps * 8 * 2 * 128 * n_tile * 32 / best / 1e9, 1),
               cycles_per_mma_at_1965MHz=round(best * 1e-3 * 1.965e9 / (reps * 8), 1))


if __name__ == "__main__":
    main()
