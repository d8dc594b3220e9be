"""Posterior sample fields behind the C ABI (csrc/svgp_step.cu: npgp_svgp_sample_prepare / npgp_svgp_sample, through
SVGPGibbs.sample): the draws against mean + K P^T Ls E + sqrt(r) xi formed in FP64 from regenerated normals, the T-only digit
contraction npgp_o8_gemm_digits, the first two moments of many draws, the invariances the Philox keys promise, the plan-state
rules, CUDA-graph capture, and a C program that trains and then draws through include/npgp.h."""
import ctypes
import math
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

from test_svgp_predict_gpu import B, CASES, N_ROWS, ROOT, build, rel

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def normals(n, seed, offset):
    """n standard normals normal_from_index(seed, offset + i), regenerated through npgp_dsvi_sample (mu 0, var 1)."""
    from nonstationary_precip_b200 import ops
    return ops.dsvi_sample(torch.zeros(n, device="cuda"), torch.ones(n, device="cuda"), seed=seed, offset=offset)


def posterior_parts(model, x, S, seed, chunk=B):
    """FP64 pieces of the draws at rows x from the factors of the plan's last prepare: predictive mean and var_f, K(x, Z),
    W = P^T Ls E, q = k^T P^T P k and the normals xi (S, n)."""
    ent = model._plan(chunk, 1, chunk)
    r = model.predictive(x, field=True, chunk=chunk)
    M, n = model.M, x.shape[0]
    P = model._plan_view(ent, 2, M * M).view(M, M).clone()
    s = torch.nn.functional.softplus(model.p["raw_outputscale"])
    K = model._kernel_fwd(x, r.field, model.p["Z"], model._field_z(), s)
    E = torch.stack([normals(M, seed, j << 32) for j in range(S)], 1)
    W = P.T @ (torch.tril(model.p["Ls"]) @ E)
    q = ((K @ P.T) ** 2).sum(1)
    xi = torch.stack([normals(n, seed, (1 << 63) + (j << 48)) for j in range(S)])
    return dict(r=r, K=K, W=W, q=q, xi=xi, s=s, P=P)


@pytest.mark.parametrize("variant,d,M", CASES)
def test_draws_equal_the_fp64_construction(variant, d, M):
    model, x, y, Z, p = build(variant, d, M, seed=M + d + 5)
    S, seed = 24, 1234
    pp = posterior_parts(model, x, S, seed)
    noise = 1e-4 + torch.nn.functional.softplus(model.p["raw_noise"])
    base = (pp["s"] + model.jitter_xx - pp["q"]).clamp_min(0.0)
    assert (base > 0).all()  # r >= jitter_xx up to rounding: no clamp here
    KW = (pp["K"] @ pp["W"]).T
    qscale = ((pp["K"].abs() @ pp["P"].abs().T) ** 2).sum(1)
    scale = (pp["K"].abs() @ pp["W"].abs()).T
    for with_noise in (False, True):
        got = model.sample(x, S, seed=seed, noise=with_noise, chunk=B)
        assert got.shape == (S, N_ROWS) and torch.isfinite(got).all()
        sd = torch.sqrt(base + noise) if with_noise else torch.sqrt(base)
        want = pp["r"].mean + KW + sd * pp["xi"]
        # K W on the tensor cores from the fixed-point planes of K and W^T: the rounding bound of the digit product, relative
        # to sum_j |K_ij||W_js|.  r = s + jitter_xx - k^T G k cancels: q is exact to eps times sum_l (sum_j |P_lj||K_ij|)^2 (the
        # size of the terms of k^T P^T P k), which sqrt(r) divides by 2 sqrt(r)
        bound = 1e-12 * scale + (1e-12 * qscale / (2 * sd) + 1e-14 * sd) * pp["xi"].abs() + 1e-15 * pp["r"].mean.abs()
        err = (got - want).abs()
        assert (err <= bound).all(), (err / bound).max().item()


@pytest.mark.parametrize("N", [64, 192])
def test_gemm_digits_against_the_decoded_planes(N):
    from nonstationary_precip_b200 import ops
    from nonstationary_precip_b200._lib import check, lib
    from test_digits_gpu import decode_planes, fwd_both, gibbs_inputs
    for variant, n, M in [("full", 300, 128), ("diag", 1000, 256), ("full", 4100, 1024)]:
        x, f1, z, f2, s, u = gibbs_inputs(variant, n, M, 3, seed=n + M + N)
        K, Ku, digits, parts = fwd_both(variant, x, f1, z, f2, s, u)
        g = torch.Generator().manual_seed(N + M)
        Bm = (torch.randn(N, M, generator=g) * torch.exp(2 * torch.randn(N, 1, generator=g))).cuda()  # row scales vary
        Bd = torch.empty(ops.digits_bytes(N, M, 64), dtype=torch.uint8, device="cuda")
        bexp = torch.empty(N, dtype=torch.int32, device="cuda")
        ops.o8_slice_rows(Bm, 64, Bd, bexp)
        ldt = N + 2
        T = torch.full((n, ldt), float("nan"), device="cuda")
        check(lib().npgp_o8_gemm_digits(n, N, M, digits.data_ptr(), None, s.data_ptr(), Bd.data_ptr(), bexp.data_ptr(),
                                        T.data_ptr(), ldt, torch.cuda.current_stream().cuda_stream), "npgp_o8_gemm_digits")
        assert T[:, N:].isnan().all()  # nothing beyond the N output columns
        T = T[:, :N]
        e = math.frexp(0.644 * 1.0000000001)[1]
        Kq = decode_planes(digits, n, M)[:n] * 2.0 ** (e - 54)
        # as test_rowquad_and_syrk_from_digits: FP64 roundings of the reference plus the dropped digit products
        trunc = 16 * math.sqrt(M) * 2.0 ** -54 * 2.0 ** e * 2 * Bm.abs().max(1).values[None, :]
        assert ((T - Kq @ Bm.T).abs() <= 1e-14 * (Kq.abs() @ Bm.abs().T) + trunc).all()
        T2 = torch.empty(n, N, device="cuda")
        check(lib().npgp_o8_gemm_digits(n, N, M, digits.data_ptr(), None, s.data_ptr(), Bd.data_ptr(), bexp.data_ptr(),
                                        T2.data_ptr(), N, torch.cuda.current_stream().cuda_stream), "npgp_o8_gemm_digits")
        assert torch.equal(T, T2)
    a = digits.data_ptr()
    assert lib().npgp_o8_gemm_digits(n, 96, M, a, None, a, a, a, a, 96, None) == -2  # N % 64
    assert lib().npgp_o8_gemm_digits(n, 64, M, a, None, a, a, a, a, 62, None) == -2  # ldt < N
    assert lib().npgp_o8_gemm_digits(n, 64, M, a, None, a, a, a, None, 64, None) == -1


@pytest.mark.parametrize("variant,d,M", [CASES[0], CASES[3]])
def test_moments_of_many_draws(variant, d, M):
    model, x, y, Z, p = build(variant, d, M, seed=31)
    x0 = x[5]
    offs = torch.tensor([0.0, 0.01, 0.03, 0.1, 0.3], device="cuda")
    xs = torch.cat([x0 + offs[:, None] * torch.ones(1, d, device="cuda"), x[100:103]]).contiguous()
    n = xs.shape[0]
    draws = torch.cat([model.sample(xs, 1024, seed=100 + k, chunk=B) for k in range(8)])  # (8192, n)
    N = draws.shape[0]
    pp = posterior_parts(model, xs, 1, 0)
    mean, var = pp["r"].mean, pp["r"].var
    A = pp["P"] @ pp["K"].T  # (M, n)
    Ls = torch.tril(model.p["Ls"])
    resid = (pp["s"] + model.jitter_xx - pp["q"]).clamp_min(0.0)
    cov = A.T @ (Ls @ Ls.T) @ A + torch.diag(resid)
    assert rel(torch.diagonal(cov), var) <= 1e-8  # each marginal is var_f (no clamp active)
    avg = draws.mean(0)
    assert ((avg - mean).abs() <= 6 * torch.sqrt(var / N)).all()
    dev = draws - avg
    emp = dev.T @ dev / (N - 1)
    band = 6 * torch.sqrt((var[:, None] * var[None, :] + cov ** 2) / (N - 1))  # sd of a sample covariance
    assert ((emp - cov).abs() <= band).all(), ((emp - cov).abs() / band).max().item()
    # nearby rows are strongly correlated in the draws: the fields are coherent, not independent marginals
    corr = cov[0, 1] / torch.sqrt(cov[0, 0] * cov[1, 1])
    assert corr > 0.5


@pytest.mark.parametrize("variant,d,M", CASES[1:3])
def test_seeds_sample_counts_row_offsets_and_chunks(variant, d, M):
    from nonstationary_precip_b200._lib import lib, ptr, stream
    model, x, y, Z, p = build(variant, d, M, seed=17)
    a = model.sample(x, 64, seed=5, chunk=B)
    assert torch.equal(a, model.sample(x, 64, seed=5, chunk=B))
    other = model.sample(x, 64, seed=6, chunk=B)
    assert not (other == a).any()
    assert torch.equal(model.sample(x, 16, seed=5, chunk=B), a[:16])
    assert torch.equal(model.sample(x, 100, seed=5, chunk=B)[:64], a)  # 128 padded rows of W^T instead of 64
    # two calls with row offsets on one prepared sampler: the rows of one call, bitwise
    ent = model._plan(B, 1, B)
    nb = lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(ent["cfg"]), 64)
    work = torch.empty(nb // 8 + 64, device="cuda")
    wp = work.data_ptr() + (-work.data_ptr()) % 256
    out = torch.full((64, N_ROWS), float("nan"), device="cuda")
    assert lib().npgp_svgp_predict_prepare(ent["handle"], ptr(model.theta), ptr(model.status), stream()) == 0
    assert lib().npgp_svgp_sample_prepare(ent["handle"], ptr(model.theta), 64, 5, wp, nb, stream()) == 0
    h = 1000  # not a chunk boundary: the chunks of the second call start elsewhere
    for lo, hi in ((0, h), (h, N_ROWS)):
        xs = x[lo:hi].contiguous()
        assert lib().npgp_svgp_sample(ent["handle"], hi - lo, ptr(xs), lo, ptr(model.theta), 0, out[:, lo:].data_ptr(), N_ROWS,
                                      wp, nb, stream()) == 0
    # mean_i is added from K u partials whose column split depends on the chunk's row count; K W, k^T G k and xi do not.  So
    # the draws are bitwise equal wherever the two chunkings give the same mean, and within the rounding of the mean elsewhere
    mean_a = model.predictive(x, chunk=B).mean
    mean_h = torch.cat([model.predictive(x[:h], chunk=B).mean, model.predictive(x[h:], chunk=B).mean])
    same = mean_a == mean_h
    assert same.float().mean() > 0.5
    assert torch.equal(out[:, same], a[:, same]) and rel(out, a) <= 1e-13
    c = model.sample(x, 64, seed=5, chunk=512)
    same = model.predictive(x, chunk=512).mean == mean_a
    assert same.float().mean() > 0.5
    assert torch.equal(c[:, same], a[:, same]) and rel(c, a) <= 1e-13


def test_plan_state_rules_and_prediction_unchanged_by_sampling():
    from nonstationary_precip_b200._lib import lib, ptr, stream
    model, x, y, Z, p = build("full", 3, 128, seed=11)
    model.use_c_engine()
    ent = model._plan(B, 1, B)
    h, th, st = ent["handle"], ptr(model.theta), stream()
    nb = lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(ent["cfg"]), 8)
    work = torch.empty(nb // 8 + 64, device="cuda")
    wp = work.data_ptr() + (-work.data_ptr()) % 256
    out = torch.empty(8, N_ROWS, device="cuda")
    xb, yb = x[:B].contiguous(), y[:B].contiguous()
    draw = lambda w=wp: lib().npgp_svgp_sample(h, N_ROWS, ptr(x), 0, th, 0, ptr(out), N_ROWS, w, nb, st)
    prep = lambda: lib().npgp_svgp_sample_prepare(h, th, 8, 3, wp, nb, st)
    assert prep() == -1 and draw() == -1  # nothing prepared yet
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    assert draw() == -1  # predict_prepare alone is not enough
    assert lib().npgp_svgp_sample_prepare(h, th, 0, 3, wp, nb, st) == -1
    assert lib().npgp_svgp_sample_prepare(h, th, 8, 3, wp, nb - 256, st) == -3
    assert prep() == 0 and draw() == 0
    assert draw(wp + 256) == -1  # another work buffer than the prepared one
    assert lib().npgp_svgp_sample(h, N_ROWS, ptr(x), 0, th, 0, ptr(out), N_ROWS - 1, wp, nb, st) == -1  # ldo < n
    first = out.clone()
    assert lib().npgp_svgp_set_extra_jitter(h, 0.0) == 0
    assert draw() == -1 and prep() == -1
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0 and prep() == 0 and draw() == 0
    assert torch.equal(out, first)
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    assert draw() == -1  # a new prepare needs a new sample_prepare
    assert lib().npgp_svgp_elbo_fwd(h, ptr(xb), ptr(yb), th, ptr(model.grad), None, st) == 0
    assert prep() == -1 and draw() == -1
    assert lib().npgp_svgp_elbo_bwd(h, ptr(xb), th, ptr(model.grad), st) == 0
    # sampling leaves P, C and their planes alone: prediction after a sample equals prediction before it, bitwise
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    mean, var = torch.empty(N_ROWS, device="cuda"), torch.empty(N_ROWS, device="cuda")
    pred = lambda: lib().npgp_svgp_predict(h, N_ROWS, ptr(x), None, th, ptr(mean), ptr(var), None, None, None, None, st)
    assert pred() == 0
    before = (mean.clone(), var.clone())
    assert prep() == 0 and draw() == 0
    assert lib().npgp_svgp_elbo_bwd(h, ptr(xb), th, ptr(model.grad), st) == -1  # the forward is invalidated
    assert pred() == 0
    assert torch.equal(mean, before[0]) and torch.equal(var, before[1])
    assert draw() == 0 and torch.equal(out, first)  # and predict does not disturb the prepared sampler


@pytest.mark.parametrize("variant", ["diag", "full"])
def test_sample_prepare_and_sample_capture_into_a_graph(variant):
    from nonstationary_precip_b200._lib import lib, ptr, stream
    model, x, y, Z, p = build(variant, 3, 128, seed=13)
    x2 = x.flip(0).contiguous() * 0.9
    want = model.sample(x2, 40, seed=9, noise=True, chunk=B)
    ent = model._plan(B, 1, B)
    nb = lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(ent["cfg"]), 40)
    work = torch.empty(nb // 8 + 64, device="cuda")
    wp = work.data_ptr() + (-work.data_ptr()) % 256
    xs = torch.zeros_like(x)
    out = torch.empty(40, N_ROWS, device="cuda")
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        assert lib().npgp_svgp_predict_prepare(ent["handle"], ptr(model.theta), ptr(model.status), stream()) == 0
        assert lib().npgp_svgp_sample_prepare(ent["handle"], ptr(model.theta), 40, 9, wp, nb, stream()) == 0
        assert lib().npgp_svgp_sample(ent["handle"], N_ROWS, ptr(xs), 0, ptr(model.theta), 1, ptr(out), N_ROWS, wp, nb,
                                      stream()) == 0
    for t in (x, x2):  # replay on other rows first, then the rows of the eager call
        xs.copy_(t)
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)


def build_demo(tmp_path):
    exe = str(tmp_path / "svgp_sample_demo")
    libdir = os.path.join(ROOT, "nonstationary_precip_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cmd = ["gcc", "-O2", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tools", "c_demo", "svgp_sample_demo.c"), "-o", exe, "-L", libdir, "-lnpgp",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm", "-Wl,-rpath," + libdir]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


@pytest.mark.parametrize("variant", ["full", "diag"])
def test_c_program_trains_then_draws(variant, tmp_path):
    exe = build_demo(tmp_path)
    M, d, iters, n, S = 128, 3, 3, N_ROWS, 256
    model, xt, yt, Z, p = build(variant, d, M, seed=29, n=n)
    x, y = xt[:B].contiguous(), yt[:B].contiguous()
    model.use_c_engine()
    consts = ([model.row_os.reshape(-1), model.row_lam.reshape(-1)] if variant == "full" else
              [model.prior_c.reshape(-1), model.prior_os.reshape(-1), model.prior_lam.reshape(-1)])
    blob = torch.cat([t.detach().reshape(-1).cpu() for t in [x, y, model.theta, model.mask] + consts]).numpy()
    prob, out = str(tmp_path / "problem.bin"), str(tmp_path / "out.bin")
    with open(prob, "wb") as f:
        f.write(struct.pack("8i", 1 if variant == "full" else 0, d, M, B, model.N, 1, 1, iters))
        f.write(blob.astype(np.float64).tobytes())
        f.write(struct.pack("i", n))
        f.write(torch.cat([xt.reshape(-1), yt]).cpu().numpy().astype(np.float64).tobytes())
    r = subprocess.run([exe, prob, out, str(S), "77"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert "finite" in r.stdout and "NOT finite" not in r.stdout
    got = np.fromfile(out, dtype=np.float64)
    n_pad = model.theta.numel()
    assert got.size == 2 * n + S * n + n_pad
    mean, var, draws, theta = np.split(got, np.cumsum([n, n, S * n]))
    draws = draws.reshape(S, n)
    assert np.isfinite(draws).all()
    # the predictive mean at the C program's theta, through Python on a plan of the same shape
    model.theta.copy_(torch.from_numpy(theta))
    want = model.predictive(xt, chunk=B)
    assert float(np.abs(mean - want.mean.cpu().numpy()).max() / np.abs(want.mean.cpu().numpy()).max()) <= 1e-12
    assert (np.abs(draws.mean(0) - mean) <= 6 * np.sqrt(var / S)).all()
    assert np.array_equal(draws, model.sample(xt, S, seed=77, chunk=B).cpu().numpy())
