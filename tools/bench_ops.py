#!/usr/bin/env python3
"""Per-kernel timings at the C2 shapes (B=65536, M=1024, d=3) with CUDA events; prints one JSON object per kernel.
Run on the GPU box:  python tools/bench_ops.py > gpurun_out/bench_ops.jsonl"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nonstationary_precip_b200 import ops  # noqa: E402
from nonstationary_precip_b200._lib import lib, ptr, stream, check  # noqa: E402

HBM = 6542.7
try:
    HBM = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    pass


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
    d = dict(kernel=name, ms_median=round(ms, 4), ms_best=round(best, 4), **kw)
    print(json.dumps(d), flush=True)


def main():
    torch.manual_seed(0)
    B, M, d = int(os.environ.get("B", 65536)), int(os.environ.get("M", 1024)), 3
    dev = "cuda"
    f64 = dict(dtype=torch.float64, device=dev)
    x = torch.rand(B, d, **f64) * 2 - 1
    z = torch.rand(M, d, **f64) * 2 - 1
    ell_x = torch.exp(0.1 * torch.randn(d, B, **f64)) * 0.3
    ell_z = torch.exp(0.1 * torch.randn(d, M, **f64)) * 0.3
    Hx, Hz = torch.randn(B, d, **f64), torch.randn(M, d, **f64)
    Dm = torch.diag(torch.tensor([0.6, 0.9, 0.5], **f64))
    Sx, Sz = ops.sigma_from_h_fwd(Hx, Dm), ops.sigma_from_h_fwd(Hz, Dm)
    s = torch.tensor(0.644, **f64)
    K = torch.empty(B, M, **f64)
    G = torch.randn(B, M, **f64)
    u = torch.randn(M, **f64)
    pairs = B * M

    out = torch.zeros(8, **f64)
    for mode, nm, flop_per in ((0, "dfma_peak", 256 * 16 * 2), (1, "dmma_peak", 8 * 16 * 512)):
        blocks, iters = 148 * 8, 4096
        ms, best = timeit(lambda: check(lib().npgp_fp64_peak_probe(mode, blocks, iters, ptr(out), stream()), nm))
        report(nm, ms, best, tflops=round(blocks * iters * flop_per / best / 1e9, 2))

    ms, best = timeit(lambda: ops.gibbs_diag_fwd(x, ell_x, z, ell_z, s, out=K))
    report("gibbs_diag_fwd", ms, best, GBs=round(pairs * 8 / best / 1e6, 1), frac_hbm=round(pairs * 8 / best / 1e6 / HBM, 3),
           gpair_s=round(pairs / best / 1e6, 2))
    ms, best = timeit(lambda: ops.gibbs_diag_bwd(x, ell_x, z, ell_z, s, G=G, need_dx2=True, need_dscale=True))
    report("gibbs_diag_bwd", ms, best, GBs=round(pairs * 8 / best / 1e6, 1), frac_hbm=round(pairs * 8 / best / 1e6 / HBM, 3))
    ms, best = timeit(lambda: ops.gibbs_full_fwd(x, Sx, z, Sz, 1e-5, s, out=K))
    report("gibbs_full_fwd", ms, best, GBs=round(pairs * 8 / best / 1e6, 1), frac_hbm=round(pairs * 8 / best / 1e6 / HBM, 3),
           gpair_s=round(pairs / best / 1e6, 2))
    ms, best = timeit(lambda: ops.gibbs_full_fwd(x, Sx, z, Sz, 1e-5, s, u=u, out=K))
    report("gibbs_full_fwd+Ku", ms, best, GBs=round(pairs * 8 / best / 1e6, 1))
    ms, best = timeit(lambda: ops.gibbs_full_bwd(x, Sx, z, Sz, 1e-5, s, G=G, need_dx2=True, need_dscale=True))
    report("gibbs_full_bwd", ms, best, GBs=round(pairs * 8 / best / 1e6, 1), frac_hbm=round(pairs * 8 / best / 1e6 / HBM, 3))

    lam3, os3 = torch.full((3, 3), 1.3, **f64), torch.ones(3, **f64)
    V3 = torch.randn(3, M, 1, **f64)
    ms, best = timeit(lambda: ops.rbf_matvec_fwd(x, z, lam3, os3, V3, None, True))
    report("rbf_matvec_fwd(nb=3,nv=1)", ms, best, gpair_s=round(pairs / best / 1e6, 2))
    dO = torch.randn(3, B, 1, **f64)
    ms, best = timeit(lambda: ops.rbf_matvec_bwd(x, z, lam3, os3, V3, dO))
    report("rbf_matvec_bwd(nb=3,nv=1)", ms, best, gpair_s=round(pairs / best / 1e6, 2))
    lam1, os1, V1 = torch.full((1, 3), 1.3, **f64), torch.ones(1, **f64), torch.randn(1, M, 3, **f64)
    ms, best = timeit(lambda: ops.rbf_matvec_fwd(x, z, lam1, os1, V1))
    report("rbf_matvec_fwd(nb=1,nv=3)", ms, best, gpair_s=round(pairs / best / 1e6, 2))
    dO1 = torch.randn(1, B, 3, **f64)
    ms, best = timeit(lambda: ops.rbf_matvec_bwd(x, z, lam1, os1, V1, dO1))
    report("rbf_matvec_bwd(nb=1,nv=3)", ms, best, gpair_s=round(pairs / best / 1e6, 2))

    Cm = torch.randn(M, M, **f64)
    T = torch.empty(B, M, **f64)
    Out = torch.empty(M, M, **f64)
    A1, A2 = torch.randn(M, M, **f64), torch.randn(M, M, **f64)
    ms, best = timeit(lambda: ops.rowquad(K, Cm, T=T))
    report("rowquad", ms, best, tflops=round(2 * B * M * M / best / 1e9, 2))
    ms, best = timeit(lambda: ops.wsyrk(K, None, out=Out))
    report("wsyrk", ms, best, tflops_full=round(2 * B * M * M / best / 1e9, 2), tflops_useful=round(B * M * (M + 128) / best / 1e9, 2))
    ms, best = timeit(lambda: ops.dgemm(A1, A2, C=Out))
    report("dgemm_MMM", ms, best, tflops=round(2 * M ** 3 / best / 1e9, 2))
    # the same two contractions on the int8 tensor cores (exact Ozaki split, csrc/ozaki.cu), slicing passes included
    Cs = 0.5 * (Cm + Cm.T)
    ms, best = timeit(lambda: ops.rowquad_i8(K, Cs, T=T))
    report("rowquad_i8[tcgen05, slicing included]", ms, best, fp64_equiv_tflops=round(2 * B * M * M / best / 1e9, 2))
    ms, best = timeit(lambda: ops.syrk_i8(K, out=Out))
    report("syrk_i8[tcgen05, slicing included]", ms, best, fp64_equiv_tflops_useful=round(B * M * (M + 64) / best / 1e9, 2))
    ms, best = timeit(lambda: torch.matmul(A1, A2, out=Out))
    report("cublas_dgemm_MMM(reference point)", ms, best, tflops=round(2 * M ** 3 / best / 1e9, 2))
    ms, best = timeit(lambda: torch.matmul(K, Cm, out=T), iters=5)
    report("cublas_dgemm_BMM(reference point)", ms, best, tflops=round(2 * B * M * M / best / 1e9, 2))
    ell = torch.full((3, M), 0.3, **f64)
    Kzz = ops.gibbs_diag_fwd(z, ell, z, ell) + 1e-6 * torch.eye(M, **f64)
    ms, best = timeit(lambda: ops.potrf_inv(Kzz))
    report("potrf_inv", ms, best)
    ms, best = timeit(lambda: torch.linalg.cholesky(Kzz))
    report("cusolver_potrf(reference point)", ms, best)


if __name__ == "__main__":
    main()
