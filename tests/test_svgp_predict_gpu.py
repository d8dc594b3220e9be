"""Posterior prediction behind the C ABI (csrc/svgp_step.cu: npgp_svgp_predict_prepare / npgp_svgp_predict, through
SVGPGibbs.predictive) against the kernel-by-kernel SVGPGibbs.predict, the CPU oracle and the closed forms of the test metrics;
its determinism, the plan-state rules it shares with the training step, CUDA-graph capture, the row-quadratic kernel without
T, and a C program that trains and then predicts through include/npgp.h."""
import math
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

from svgp_cases import make_problem

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 640
N_ROWS = 3 * B + 77  # three whole chunks and a ragged one
CASES = [("diag", 2, 128), ("diag", 3, 256), ("full", 3, 128), ("full", 3, 256)]


def rel(a, b):
    a, b = a.detach().cpu(), b.detach().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


def build(variant, d, M, seed, n=N_ROWS, **opts):
    from nonstationary_precip_b200.svgp import SVGPGibbs
    x, y, Z, p, N = make_problem(variant, B=n, M=M, d=d, seed=seed, device="cuda")
    return SVGPGibbs(variant, Z, N, **p, **opts), x, y, Z, p


def oracle_field(model, x, p):
    """The latent field of the oracle at rows x: ell(x) (d, n) or Sigma(x) packed as npgp_sigma_from_h_fwd (n, P)."""
    from oracle import gibbs_oracle as o
    c = lambda t: t.detach().cpu()
    x, Z = c(x), c(model.p["Z"])
    if model.variant == "diag":
        return o.field_interp_diag(x, Z, torch.exp(c(model.p["log_ell_z"])), c(p["prior_c"]), c(p["prior_os"]), c(p["prior_lam"]))
    Hx = o.field_interp_H(x, Z, c(model.p["H"]), torch.tensor(float(p["row_os"])), c(p["row_lam"]))
    S = o.sigma_from_H(Hx, c(model.p["D"]))
    iu = torch.triu_indices(model.d, model.d)
    return S[:, iu[0], iu[1]]


def oracle_predict(model, x, p):
    from oracle import gibbs_oracle as o
    from nonstationary_precip_b200.svgp import _inv_softplus
    c = lambda t: t.detach().cpu()
    extra = (dict(log_ell_z=c(model.p["log_ell_z"]), prior_c=c(p["prior_c"]), prior_os=c(p["prior_os"]),
                  prior_lam=c(p["prior_lam"])) if model.variant == "diag" else
             dict(H=c(model.p["H"]), Dm=c(model.p["D"]), row_os=torch.tensor(float(p["row_os"])), row_lam=c(p["row_lam"])))
    return o.svgp_gibbs_predict(c(x), c(model.p["Z"]), c(model.p["m"]), c(model.p["Ls"]),
                                torch.tensor(_inv_softplus(p["outputscale"])), model.variant, **extra)


def rowside_reference(model, ent, x, field):
    """mean and var_f at the rows x from the plan's Z-side factors of its last prepare (u, C) and the returned field, with the
    row-side kernels launched one by one as predict() launches them (all rows at once, sums in torch)."""
    from nonstationary_precip_b200 import ops
    M, n = model.M, x.shape[0]
    u = model._plan_view(ent, 4, M)
    Cm = model._plan_view(ent, 3, M * M).view(M, M)
    s = torch.nn.functional.softplus(model.p["raw_outputscale"])
    digits = torch.empty(ops.digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
    parts = torch.empty(ops.gibbs_digits_splits(n, M), n, device="cuda")
    model._kernel_fwd_digits(x, field, model.p["Z"], model._field_z(), s, u, dict(Ad=digits, mu_part=parts))
    Cd = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device="cuda")
    cexp = torch.empty(M, dtype=torch.int32, device="cuda")
    ops.o8_slice_rows(Cm, 64, Cd, cexp)
    q_part = torch.empty(M // 64, n, device="cuda")
    ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, None, q_part=q_part)
    return parts.sum(0), (s + model.jitter_xx + q_part.sum(0)).clamp_min(1e-6)


def c_predict(model, ent, xs, ys=None, sums=None, field=None, prepare=True):
    """Raw C calls on a plan entry of model._plan; returns (rc_prepare, rc_predict, mean, var_f, var_y, lpd)."""
    from nonstationary_precip_b200._lib import lib, ptr, stream
    n = xs.shape[0]
    mean, var, var_y = (torch.empty(n, device="cuda") for _ in range(3))
    lpd = torch.empty(n, device="cuda") if ys is not None else None
    rc0 = lib().npgp_svgp_predict_prepare(ent["handle"], ptr(model.theta), ptr(model.status), stream()) if prepare else 0
    rc1 = lib().npgp_svgp_predict(ent["handle"], n, ptr(xs), ptr(ys), ptr(model.theta), ptr(mean), ptr(var), ptr(var_y),
                                  ptr(field), ptr(lpd), ptr(sums), stream())
    return rc0, rc1, mean, var, var_y, lpd


@pytest.mark.parametrize("variant,d,M", CASES)
def test_predictive_matches_predict_oracle_and_metrics(variant, d, M):
    from nonstationary_precip_b200.utils import metrics
    model, x, y, Z, p = build(variant, d, M, seed=M + d)
    r = model.predictive(x, y, field=True, chunk=B)
    assert model.check_status() == 0
    # the chunked row side against the same Z-side factors: only the order of a few partial sums differs
    mean_r, var_r = rowside_reference(model, model._plan(B, 1, B), x, r.field)
    assert rel(r.mean, mean_r) <= 1e-12 and rel(r.var, var_r) <= 1e-12, (rel(r.mean, mean_r), rel(r.var, var_r))
    # predict() factors Kzz and solves for the field weights with other kernels (and forms C in full where the C path mirrors
    # its lower tiles): the two differ by eps * cond(Kzz), cond(K_prior), as the two training engines do
    mean_p, var_p = model.predict(x, chunk=B)
    assert rel(r.mean, mean_p) <= 1e-8 and rel(r.var, var_p) <= 1e-8, (rel(r.mean, mean_p), rel(r.var, var_p))
    mean_o, var_o = oracle_predict(model, x, p)
    assert rel(r.mean, mean_o) <= 1e-8 and rel(r.var, var_o) <= 1e-8, (rel(r.mean, mean_o), rel(r.var, var_o))
    # the oracle solves for the field weights by LU, the C path through the inverse Cholesky factor: eps * cond(K_prior)
    # apart (cond ~1e6 .. 1e7 here)
    assert rel(r.field, oracle_field(model, x, p)) <= 1e-8
    noise = 1e-4 + torch.nn.functional.softplus(model.p["raw_noise"])
    assert rel(r.var_y - r.var, noise.expand(N_ROWS)) <= 1e-13
    lpd = -0.5 * (math.log(2 * math.pi) + torch.log(r.var_y) + (y - r.mean) ** 2 / r.var_y)
    assert rel(r.lpd, lpd) <= 1e-13
    s = r.sums.cpu()
    assert s[2].item() == N_ROWS
    nlpd = metrics.negative_log_predictive_density(y, r.mean, r.var_y).item()
    assert abs(s[1].item() / N_ROWS - nlpd) <= 1e-12 * abs(nlpd)
    rmse = float(metrics.rmse(r.mean, y, 1))
    assert abs(math.sqrt(s[0].item() / N_ROWS) - rmse) <= 1e-12 * rmse


@pytest.mark.parametrize("variant,d,M", CASES[1:3])
def test_predictive_is_deterministic_and_shards(variant, d, M):
    model, x, y, Z, p = build(variant, d, M, seed=7)
    a, b = model.predictive(x, y, field=True, chunk=B), model.predictive(x, y, field=True, chunk=B)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    # rows in two calls into one zeroed sums (what a caller sharding rows over ranks does before one all-reduce)
    ent = model._plan(B, 1, B)
    sums = torch.zeros(3, device="cuda")
    h = 1000
    halves = [c_predict(model, ent, x[:h], y[:h], sums), c_predict(model, ent, x[h:], y[h:], sums, prepare=False)]
    assert all(rc0 == 0 and rc1 == 0 for rc0, rc1, *_ in halves)
    assert rel(sums, a.sums) <= 1e-14
    assert rel(torch.cat([halves[0][2], halves[1][2]]), a.mean) <= 1e-14
    assert rel(torch.cat([halves[0][3], halves[1][3]]), a.var) <= 1e-14
    # a plan with another chunk size streams the rows differently
    c = model.predictive(x, y, field=True, chunk=512)
    for u, v in zip(c, a):
        assert rel(u, v) <= 1e-13


def test_ragged_last_chunk_with_more_mean_partials_than_a_full_chunk():
    """M = 1024, 20000-row chunks: the Gibbs digits kernel splits the columns of a 20000-row chunk 4 ways, of the 15000-row last
    chunk 6 ways, so that chunk's K u partials (6 x 15000) do not fit the 4 x 20000 the plan keeps for the step."""
    from nonstationary_precip_b200._lib import lib
    assert lib().npgp_gibbs_digits_splits(20000, 1024) * 20000 < lib().npgp_gibbs_digits_splits(15000, 1024) * 15000
    model, x, y, Z, p = build("diag", 2, 1024, seed=3, n=35000)
    r = model.predictive(x, y, field=True, chunk=20000)
    mean_r, var_r = rowside_reference(model, model._plan(20000, 1, 20000), x, r.field)
    # var: the same products and partials; mean: the reference adds 4 column-split partials where the last chunk has 6, and
    # K u cancels strongly at M = 1024 (|u| >> |mean|), so the two groupings round apart by eps * sum_j |K_ij u_j|
    assert rel(r.var, var_r) <= 1e-12 and rel(r.mean, mean_r) <= 1e-10, (rel(r.var, var_r), rel(r.mean, mean_r))
    assert r.sums[2].item() == 35000


def test_plan_state_rules_and_training_unchanged_by_prediction():
    from nonstationary_precip_b200._lib import lib, ptr, stream
    ma, x, y, Z, p = build("full", 3, 128, seed=11)
    mb, *_ = build("full", 3, 128, seed=11)
    ma.use_c_engine()
    mb.use_c_engine()
    xb, yb = x[:B].contiguous(), y[:B].contiguous()
    ent = ma._plan(B, 1, B)
    assert c_predict(ma, ent, x, prepare=False)[1] == -1  # no prepare yet
    assert lib().npgp_svgp_elbo_fwd(ent["handle"], ptr(xb), ptr(yb), ptr(ma.theta), ptr(ma.grad), None, stream()) == 0
    assert c_predict(ma, ent, x)[:2] == (0, 0)
    assert lib().npgp_svgp_elbo_bwd(ent["handle"], ptr(xb), ptr(ma.theta), ptr(ma.grad), stream()) == -1  # fwd overwritten
    assert lib().npgp_svgp_set_extra_jitter(ent["handle"], 0.0) == 0
    assert c_predict(ma, ent, x, prepare=False)[1] == -1
    assert c_predict(ma, ent, x)[:2] == (0, 0)
    la, lb = [], []
    for k in range(3):
        la.append(ma.train_step(xb, yb, lr=0.01).item())
        assert c_predict(ma, ent, x, prepare=False)[1] == -1  # a step invalidates the prepared factors
        assert c_predict(ma, ent, x, y)[:2] == (0, 0)
        lb.append(mb.train_step(xb, yb, lr=0.01).item())
    # the forward is fixed-order: the first loss is bitwise; the backward accumulates with FP64 atomics, which Adam carries into
    # the later steps of two runs with or without prediction alike
    assert la[0] == lb[0]
    for u, v in zip(la, lb):
        assert abs(u - v) <= 1e-10 * abs(v)
    assert rel(ma.theta, mb.theta) <= 1e-8 and ma.check_status() == 0  # as test_svgp_cstep_gpu.py
    # no trace of the prediction in the plan: at one theta, its forward equals that of the plan that never predicted
    ma.theta.copy_(mb.theta)
    for m in (ma, mb):
        e = m._plan(B, 1, B)
        assert lib().npgp_svgp_elbo_fwd(e["handle"], ptr(xb), ptr(yb), ptr(m.theta), ptr(m.grad), None, stream()) == 0
    assert ma.grad[-2].item() == mb.grad[-2].item()


@pytest.mark.parametrize("variant", ["diag", "full"])
def test_prepare_and_predict_capture_into_a_graph(variant):
    from nonstationary_precip_b200._lib import lib, ptr, stream
    model, x, y, Z, p = build(variant, 3, 128, seed=13)
    x2, y2 = x.flip(0).contiguous() * 0.9, y.flip(0).contiguous()
    ent = model._plan(B, 1, B)
    want = model.predictive(x2, y2, field=True, chunk=B)
    xs, ys = torch.zeros_like(x), torch.zeros_like(y)
    outs = [torch.empty_like(t) for t in want]
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs[5].zero_()
        assert lib().npgp_svgp_predict_prepare(ent["handle"], ptr(model.theta), ptr(model.status), stream()) == 0
        assert lib().npgp_svgp_predict(ent["handle"], N_ROWS, ptr(xs), ptr(ys), ptr(model.theta), *[ptr(t) for t in outs],
                                       stream()) == 0
    for t in (x, x2):  # replay on other rows first, then the rows of the eager call
        xs.copy_(t)
        ys.copy_(y2)
        graph.replay()
    torch.cuda.synchronize()
    for u, v in zip(outs, want):
        assert torch.equal(u, v)


def test_rowquad_without_t_gives_the_same_q():
    from nonstationary_precip_b200 import ops
    from nonstationary_precip_b200._lib import lib
    from test_digits_gpu import fwd_both, gibbs_inputs
    for variant, n, M in [("full", 300, 128), ("full", 4100, 1024), ("diag", 2000, 256)]:
        x, f1, z, f2, s, u = gibbs_inputs(variant, n, M, 3, seed=7 * n + M)
        K, Ku, digits, parts = fwd_both(variant, x, f1, z, f2, s, u)
        g = torch.Generator().manual_seed(3)
        A = torch.randn(M, M, generator=g).cuda()
        Cm = A @ A.T / M - 0.3 * torch.eye(M, device="cuda")
        Cm = 0.5 * (Cm + Cm.T)
        Cd = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device="cuda")
        cexp = torch.empty(M, dtype=torch.int32, device="cuda")
        ops.o8_slice_rows(Cm, 64, Cd, cexp)
        T = torch.empty(n, M, device="cuda")
        q1 = torch.full((M // 64, n), float("nan"), device="cuda")
        q2 = torch.full((M // 64, n), float("nan"), device="cuda")
        ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, T, q_part=q1)
        assert ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, None, q_part=q2) is None
        assert torch.equal(q1, q2)
    a = digits.data_ptr()
    assert lib().npgp_o8_rowquad_digits(n, M, a, None, s.data_ptr(), a, a, None, 0, None, M, None, 0, None, None, None) == -1


def test_prepare_flags_an_indefinite_kzz():
    model, x, y, Z, p = build("diag", 3, 128, seed=3, jitter_zz=-1.0)
    model.predictive(x, chunk=B)
    assert model.check_status() & 1


def build_demo(tmp_path):
    exe = str(tmp_path / "svgp_predict_demo")
    libdir = os.path.join(ROOT, "nonstationary_precip_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cmd = ["gcc", "-O2", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tools", "c_demo", "svgp_predict_demo.c"), "-o", exe, "-L", libdir, "-lnpgp",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm", "-Wl,-rpath," + libdir]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


@pytest.mark.parametrize("variant", ["full", "diag"])
def test_c_program_trains_then_predicts_like_predictive(variant, tmp_path):
    exe = build_demo(tmp_path)
    M, d, iters, n = 128, 3, 3, N_ROWS
    model, xt, yt, Z, p = build(variant, d, M, seed=23, n=n)
    x, y = xt[:B].contiguous(), yt[:B].contiguous()
    N = model.N
    model.use_c_engine()
    consts = ([model.row_os.reshape(-1), model.row_lam.reshape(-1)] if variant == "full" else
              [model.prior_c.reshape(-1), model.prior_os.reshape(-1), model.prior_lam.reshape(-1)])
    blob = torch.cat([t.detach().reshape(-1).cpu() for t in [x, y, model.theta, model.mask] + consts]).numpy()
    prob, out = str(tmp_path / "problem.bin"), str(tmp_path / "out.bin")
    with open(prob, "wb") as f:
        f.write(struct.pack("8i", 1 if variant == "full" else 0, d, M, B, N, 1, 1, iters))
        f.write(blob.astype(np.float64).tobytes())
        f.write(struct.pack("i", n))
        f.write(torch.cat([xt.reshape(-1), yt]).cpu().numpy().astype(np.float64).tobytes())
    r = subprocess.run([exe, prob, out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.stdout, r.stderr)
    for _ in range(iters):
        model.train_step(x, y, lr=0.01)
    got = np.fromfile(out, dtype=np.float64)
    P = d if variant == "diag" else d * (d + 1) // 2
    n_pad = model.theta.numel()
    assert got.size == 4 * n + n * P + 3 + n_pad
    parts = np.split(got, np.cumsum([n, n, n, n * P, n, 3]))
    rel_np = lambda a, b: float(np.abs(a - b).max() / np.abs(b).max())
    # the same steps (to the FP64 atomics of the backward, as in test_c_caller_gpu.py), then the prediction at the C program's
    # theta: the same calls on the same plan shape
    assert rel_np(parts[6], model.theta.cpu().numpy()) <= 1e-8
    model.theta.copy_(torch.from_numpy(parts[6]))
    want = model.predictive(xt, yt, field=True, chunk=B)
    for g, w in zip(parts, [want.mean, want.var, want.var_y, want.field.reshape(-1), want.lpd, want.sums]):
        assert rel_np(g, w.cpu().numpy()) <= 1e-9
