"""The whole SVGP-Gibbs ELBO step behind the C ABI (csrc/svgp_step.cu: npgp_svgp_elbo_fwd / _bwd / npgp_svgp_step) against the
CPU oracle and against the kernel-by-kernel Python orchestration of the same step (nonstationary_precip_b200/svgp.py)."""
import pytest
import torch

from svgp_cases import make_problem, oracle_loss_and_grads

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def rel(a, b):
    a, b = a.detach().cpu(), b.detach().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


def build(variant, engine, **kw):
    from nonstationary_precip_b200.svgp import SVGPGibbs
    opts = {k: kw.pop(k) for k in ("learn_inducing_locations", "include_prior", "jitter_zz") if k in kw}
    x, y, Z, p, N = make_problem(variant, device="cuda", **kw)
    model = SVGPGibbs(variant, Z, N, **p, **opts)
    if engine == "c":
        model.use_c_engine()
    return model, x, y, Z, p, N


@pytest.mark.parametrize("variant,d,B,M", [("full", 3, 700, 128), ("full", 2, 513, 256), ("diag", 3, 700, 128),
                                            ("diag", 2, 300, 256)])
def test_c_step_matches_oracle_and_python_engine(variant, d, B, M):
    mc, x, y, Z, p, N = build(variant, "c", B=B, M=M, d=d, seed=1)
    mp, *_ = build(variant, "python", B=B, M=M, d=d, seed=1)
    loss_c = mc.loss_and_grad(x, y)
    loss_p = mp.loss_and_grad(x, y)
    assert int(mc.last["info"]) == 0 and mc.check_status() == 0
    want_loss, want = oracle_loss_and_grads(variant, x, y, Z, p, N)
    # north_star tolerance: ELBO within 1e-6 relative
    assert abs(loss_c.item() - want_loss.item()) < 1e-9 * abs(want_loss.item())
    for name, gw in want.items():
        assert rel(mc.g[name], gw) < 1e-6, name
    # the two orchestrations launch the same kernels on the same data: they agree far below the oracle tolerance
    # (C = P^T E P is mirrored from its lower tiles in the C step and computed in full by the Python orchestration: the two
    # differ by eps * cond(Kzz), like either of them from the oracle)
    assert abs(loss_c.item() - loss_p.item()) < 1e-8 * abs(loss_p.item())
    for name in mp.g:
        assert rel(mc.g[name], mp.g[name]) < 1e-7, name  # FP64 atomics in both engines; the oracle bound above is the parity claim
    assert rel(mc.last["mu"], mp.last["mu"]) < 1e-8  # (the engines solve K_row W = H with different kernels: cond(K_row) eps)


@pytest.mark.parametrize("variant", ["full", "diag"])
@pytest.mark.parametrize("opts", [dict(learn_inducing_locations=False), dict(include_prior=False)])
def test_c_step_options(variant, opts):
    mc, x, y, Z, p, N = build(variant, "c", B=400, M=128, d=3, seed=2, **opts)
    mp, *_ = build(variant, "python", B=400, M=128, d=3, seed=2, **opts)
    lc, lp = mc.loss_and_grad(x, y, world_size=2), mp.loss_and_grad(x, y, world_size=2)
    frozen_z = opts.get("learn_inducing_locations") is False
    # this rank's share with B_global = 2 B and the replicated terms weighted 1/2 is half the one-rank -ELBO of (x, y)
    want_loss, want = oracle_loss_and_grads(variant, x, y, Z, p, N, include_prior=opts.get("include_prior", True),
                                            learn_z=not frozen_z)
    assert abs(2 * lc.item() - want_loss.item()) < 1e-9 * abs(want_loss.item())
    for name, gw in want.items():
        if name == "Z" and frozen_z:
            continue  # frozen by the Adam mask; the engines need not agree on the unused slot
        assert rel(2 * mc.g[name], gw) < 1e-6, name  # the north-star bound of the test above
    assert abs(lc.item() - lp.item()) < 1e-8 * abs(lp.item())
    for name in mp.g:
        if name == "Z" and frozen_z:
            continue
        assert rel(mc.g[name], mp.g[name]) < 1e-7, name  # FP64 atomics in both engines; the oracle bound above is the parity claim


@pytest.mark.parametrize("variant", ["full", "diag"])
def test_c_train_steps_eager_and_graph_match_python_engine(variant):
    mc, x, y, Z, p, N = build(variant, "c", B=512, M=128, d=3, seed=4)
    mg, *_ = build(variant, "c", B=512, M=128, d=3, seed=4)
    mp, *_ = build(variant, "python", B=512, M=128, d=3, seed=4)
    mg.capture(512, 1, 512, lr=0.01)
    for _ in range(4):
        lc = mc.train_step(x, y, lr=0.01)  # one C call: npgp_svgp_step
        lg = mg.train_step_graph(x, y)     # the same call replayed from a CUDA graph
        lp = mp.train_step(x, y, lr=0.01)
        assert abs(lc.item() - lp.item()) < 1e-9 * abs(lp.item())
        assert abs(lg.item() - lp.item()) < 1e-9 * abs(lp.item())
    assert rel(mc.theta, mp.theta) < 1e-8 and rel(mg.theta, mp.theta) < 1e-8
    assert float(mc.step_dev) == 4.0 and float(mg.step_dev) == 4.0 and mc.check_status() == 0


def test_c_step_rows_shard_linearly():
    """Two half batches with the replicated terms weighted 1/2 sum to the full-batch gradient (what the all-reduce relies on)."""
    mc, x, y, Z, p, N = build("full", "c", B=1024, M=128, d=3, seed=5)
    mc.loss_and_grad(x, y)
    g_full = mc.grad.clone()
    tot = torch.zeros_like(g_full)
    for r in range(2):
        mc.loss_and_grad(x[r::2].contiguous(), y[r::2].contiguous(), world_size=2, B_global=1024)
        tot += mc.grad
    assert rel(tot, g_full) < 1e-9


def test_c_step_failed_cholesky_is_flagged_and_guarded():
    mc, x, y, Z, p, N = build("diag", "c", B=512, M=128, d=3, seed=3, jitter_zz=-1.0)
    before = mc.theta.clone()
    for _ in range(2):
        mc.train_step(x, y, lr=0.01)
    assert mc.check_status() & 1
    assert torch.equal(mc.theta, before) and float(mc.step_dev) == 0.0
    # the ladder is driven from the host: more jitter does not repair -1.0, and the last rung raises
    for _ in range(3):
        mc.recover()
        mc.train_step(x, y, lr=0.01)
        assert mc.check_status() & 1
    with pytest.raises(RuntimeError):
        mc.recover()


def test_c_step_argument_errors():
    import ctypes as C
    from nonstationary_precip_b200._lib import SvgpConfig, lib
    cfg = SvgpConfig(variant=1, d=3, M=100, B_local=64, N_total=1000, B_global=64, world_size=1)
    assert lib().npgp_svgp_workspace_bytes(C.byref(cfg)) == -1  # M % 128 != 0
    cfg = SvgpConfig(variant=1, d=4, M=128, B_local=64, N_total=1000, B_global=64, world_size=1)
    assert lib().npgp_svgp_workspace_bytes(C.byref(cfg)) == -1  # the full-matrix kernel is closed form for d = 2, 3 only
    cfg = SvgpConfig(variant=0, d=3, M=128, B_local=64, N_total=1000, B_global=64, world_size=1)
    assert lib().npgp_svgp_workspace_bytes(C.byref(cfg)) > 0
    handle = C.c_void_p()
    ws = torch.empty(1024, dtype=torch.uint8, device="cuda")
    assert lib().npgp_svgp_plan_create(C.byref(handle), C.byref(cfg), ws.data_ptr(), 1024) == -1  # prior constants missing


def test_npgp_comm_single_rank_allreduce():
    """npgp_comm_* / npgp_allreduce_f64 on a one-rank communicator (NCCL bound at run time): identity, capturable."""
    from nonstationary_precip_b200.comm import NpgpComm
    comm = NpgpComm(0, 1, torch.device("cuda", 0))
    t = torch.arange(1000, dtype=torch.float64, device="cuda")
    comm(t)
    torch.cuda.synchronize()
    assert torch.equal(t.cpu(), torch.arange(1000, dtype=torch.float64))
    comm.destroy()


@pytest.mark.parametrize("engine", ["c", "python"])
def test_pipelined_graph_replay_equals_sequential_steps(engine):
    """capture(buffers=2) + train_step_graph_async / loss_result: the host-to-device copy of minibatch k + 1 runs under step k and
    the loss of step k is read while step k + 1 runs; results equal the plain step-by-step loop on the same minibatches."""
    ma, x, y, Z, p, N = build("full", engine, B=2048, M=128, d=3, seed=6)
    mb, *_ = build("full", engine, B=2048, M=128, d=3, seed=6)
    xs, ys = x.cpu().pin_memory(), y.cpu().pin_memory()
    ma.capture(512, 1, 512, lr=0.01, buffers=2)
    got, prev = [], None
    for k in range(4):
        t = ma.train_step_graph_async(xs[512 * k:512 * (k + 1)], ys[512 * k:512 * (k + 1)])
        if prev is not None:
            got.append(ma.loss_result(prev))
        prev = t
    got.append(ma.loss_result(prev))
    want = [mb.train_step(x[512 * k:512 * (k + 1)].contiguous(), y[512 * k:512 * (k + 1)].contiguous(), lr=0.01).item()
            for k in range(4)]
    for a, b in zip(got, want):
        assert abs(a - b) < 1e-9 * abs(b)
    assert rel(ma.theta, mb.theta) < 1e-8 and float(ma.step_dev) == 4.0
