"""Whitened SVGP with a Gibbs prior covariance whose latent lengthscale field lives at the inducing points -- the
"SVGP-Gibbs ELBO" of BASELINE.json (composition defined in SURVEY.md Appendix B from the reference's parts:
InducingGibbsKernel's field handling, models/gibbs_kernels.py:210-223; the multivariate kernels,
models/sparse_multivariate_gibbs_kernel.py:67-154; GPyTorch's whitened VariationalStrategy + VariationalELBO as driven
by models/dgps.py:25-35 and experiments/deepgp_spatial_bench.py:61,84-87).

One training step = field interpolation -> K(X_B,Z), Kzz -> Cholesky -> whitened predictive mean/variance ->
Gaussian E[log-lik] + KL -> ANALYTIC backward (no autograd graph) -> one all-reduce of the flat gradient -> Adam.
Every O(B*M), O(B*M^2) and O(M^3) operation is a hand-written kernel behind the C ABI (``ops``); torch is used for
device memory, streams, O(M^2)/O(B) elementwise glue and ``torch.distributed``.

Gradient chain used below (E = S - I, S = Ls Ls^T, P = L^-1, L = chol(Kzz + jitter I), u = P^T m, C = P^T E P):
    mu = K u,  v = s + jitter_xx + rowdot(K C, K)
    G  = dELBO/dK   = g_mu u^T + 2 diag(g_v) (K C)            (formed inside the Gibbs backward kernel)
    du = K^T g_mu,  dC = K^T diag(g_v) K,  dm = P du,  dE = P dC P^T,  dLs = tril(2 dE Ls)
    dKzz = sym( P^T Phi(-(2 E dE + m dm^T)) P )               (Cholesky + inverse backward folded: L^T dL = -dP P^T)
"""
from __future__ import annotations

import contextlib
import math
from typing import NamedTuple, Optional

import torch

from . import ops as _cuda_ops

LOG2PI = math.log(2.0 * math.pi)


def _softplus(x):
    return torch.nn.functional.softplus(x)


def _inv_softplus(v: float) -> float:
    return v + math.log(-math.expm1(-v))


class Predictive(NamedTuple):
    """Posterior marginals of SVGPGibbs.predictive at n rows: var of f, var_y = var + noise; field (field=True): ell(x) (d, n)
    for 'diag', packed Sigma(x) (n, d(d+1)/2) for 'full'; with y: lpd = log N(y | mean, var_y) (n) and
    sums = [sum (y - mean)^2, sum -lpd, n] (3), whose all-reduce over ranks gives the global RMSE / NLPD."""
    mean: torch.Tensor
    var: torch.Tensor
    var_y: torch.Tensor
    field: Optional[torch.Tensor]
    lpd: Optional[torch.Tensor]
    sums: Optional[torch.Tensor]


class _Section:
    """Bracket around a named part of the step.  model.profile (a dict): CUDA-event pairs (eager runs only).
    model.timeline (an int64 device buffer): GPU-timer stamps written by tiny kernels, which ARE capturable, so the real
    start / end of every section inside a replayed multi-stream graph can be read back (SVGPGibbs.timeline_ms)."""

    def __init__(self, model, name):
        self.model, self.name = model, name

    def __enter__(self):
        m = self.model
        if m.profile is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        if m.timeline is not None:
            self.slot = m._timeline_slots.setdefault(self.name, len(m._timeline_slots))
            m.o.timestamp(m.timeline, 2 * self.slot)
        return self

    def __exit__(self, *exc):
        m = self.model
        if m.profile is not None:
            self.b.record()
            m.profile.setdefault(self.name, []).append((self.a, self.b))
        if m.timeline is not None:
            m.o.timestamp(m.timeline, 2 * self.slot + 1)
        return False


class SVGPGibbs:
    """variant = 'diag' (GibbsKernel, log-normal field) or 'full' (multivariate Gibbs, matrix-valued field H, D)."""

    def __init__(self, variant: str, Z: torch.Tensor, N_total: int, *, log_ell_z=None, prior_c=None, prior_os=None,
                 prior_lam=None, H=None, Dm=None, row_os=None, row_lam=None, m=None, Ls=None, outputscale=0.644,
                 noise=0.011, jitter_zz=1e-6, jitter_xx=1e-4, kernel_jitter=1e-5, learn_inducing_locations=True,
                 include_prior=True, ops=None):
        assert variant in ("diag", "full")
        self.o = ops if ops is not None else _cuda_ops
        self.variant, self.N = variant, int(N_total)
        self.dev = Z.device
        self.M, self.d = Z.shape
        M, d = self.M, self.d
        self.jitter_zz, self.jitter_xx, self.kernel_jitter = jitter_zz, jitter_xx, kernel_jitter
        self.learn_z, self.include_prior = learn_inducing_locations, include_prior
        f64 = dict(dtype=torch.float64, device=self.dev)
        # ---- flat parameter / gradient buffers with named views
        shapes = [("Z", (M, d))]
        shapes += [("log_ell_z", (d, M))] if variant == "diag" else [("H", (M, d)), ("D", (d, d))]
        shapes += [("m", (M,)), ("Ls", (M, M)), ("raw_outputscale", (1,)), ("raw_noise", (1,))]
        self.shapes = shapes
        n = sum(int(torch.tensor(s).prod()) for _, s in shapes)
        n_pad = (n + 1) // 2 * 2
        self.theta = torch.zeros(n_pad, **f64)
        self.grad = torch.zeros(n_pad + 2, **f64)  # [-2]: loss, [-1]: spare -> one all-reduce carries everything
        self.adam_m, self.adam_v = torch.zeros(n_pad, **f64), torch.zeros(n_pad, **f64)
        self.mask = torch.ones(n_pad, **f64)
        self.p, self.g, self._mask_views = {}, {}, {}
        off = 0
        for name, shp in shapes:
            k = int(torch.tensor(shp).prod())
            self.p[name] = self.theta[off:off + k].view(*shp)
            self.g[name] = self.grad[off:off + k].view(*shp)
            self._mask_views[name] = self.mask[off:off + k].view(*shp)
            off += k
        self.n_params = n
        self.p["Z"].copy_(Z)
        if variant == "diag":
            self.p["log_ell_z"].copy_(log_ell_z)
            self.prior_c, self.prior_os, self.prior_lam = (t.to(**f64).contiguous() for t in (prior_c, prior_os, prior_lam))
        else:
            self.p["H"].copy_(H)
            self.p["D"].copy_(Dm)
            self.row_os = torch.as_tensor(row_os, **f64).reshape(1).contiguous()
            self.row_lam = torch.as_tensor(row_lam, **f64).reshape(1, d).contiguous()
            if not torch.allclose(Dm * Dm, (Dm * Dm).T):
                raise ValueError("D o D must be symmetric (the reference initialises D diagonal)")
        self.p["m"].copy_(m if m is not None else torch.zeros(M))
        self.p["Ls"].copy_(Ls if Ls is not None else torch.eye(M))
        self.p["raw_outputscale"].fill_(_inv_softplus(outputscale))
        self.p["raw_noise"].fill_(_inv_softplus(noise - 1e-4))
        self._mask_views["Ls"].copy_(torch.tril(torch.ones(M, M)))
        if not learn_inducing_locations:
            self._mask_views["Z"].zero_()
        self.eye = torch.eye(M, **f64)
        self.step_count = 0
        self.step_dev = torch.zeros(1, **f64)  # Adam step counter on the device
        # sticky failure flag on the device (bit 0: a Cholesky failed, bit 1: non-finite loss); the guarded Adam kernel
        # leaves the parameters alone while it is set, the host polls it (check_status) and escalates the jitter (recover)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.dev) if self.dev.type == "cuda" else None
        self.extra_jitter = 0.0  # psd_safe_cholesky ladder on top of jitter_zz: 0, 1e-8, 1e-7, 1e-6 (then raise)
        self._side = torch.cuda.Stream(device=self.dev) if self.dev.type == "cuda" else None
        self._side2 = torch.cuda.Stream(device=self.dev) if self.dev.type == "cuda" else None
        self.overlap = True
        # row-quadratic GEMM T = K C: "dmma" (FP64 tensor pipe, dgemm.cu) or "i8" (exact Ozaki split on tcgen05 int8,
        # ozaki.cu; needs M % 64 == 0).  Same result to FP64 rounding (tests/test_ozaki_gpu.py).
        self.rowquad_impl = "i8"  # falls back to "dmma" per call when M is not a multiple of 128
        self._i8_bufs = {}  # digit planes / partial buffers of the int8 path, per local batch size (owned by this model)
        # "python": the step is orchestrated below, kernel by kernel through `ops`; "c": ONE C call per pass (csrc/svgp_step.cu:
        # npgp_svgp_elbo_fwd / _bwd / npgp_svgp_step on a plan with its own workspace and side streams; digit path only)
        self.engine = "python"
        self._plans = {}
        self._graph = None
        self.profile = None  # set to a dict to collect per-section CUDA-event pairs
        self.timeline = None  # set to an int64 device buffer (>= 64 entries) to stamp section boundaries (capturable)
        self._timeline_slots = {}

    def _sec(self, name):
        return _Section(self, name)

    def timeline_ms(self):
        """{section: (start_ms, end_ms)} relative to the earliest stamp of the last replayed / executed step."""
        t = self.timeline.cpu()
        used = [v for v in t[:2 * len(self._timeline_slots)].tolist() if v > 0]
        t0 = min(used)
        return {k: (round((t[2 * s].item() - t0) / 1e6, 4), round((t[2 * s + 1].item() - t0) / 1e6, 4))
                for k, s in self._timeline_slots.items() if t[2 * s].item() > 0 and t[2 * s + 1].item() > 0}

    def section_ms(self):
        """Mean milliseconds per section from the collected events (call after torch.cuda.synchronize())."""
        return {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in (self.profile or {}).items()}

    # ------------------------------------------------------------------------------------------------------------------
    def freeze(self, name):
        self._mask_views[name].zero_()

    def state_dict(self):
        return {k: v.clone() for k, v in self.p.items()}

    def snapshot(self):
        """Parameters + optimiser state (for restarting a run from the same point)."""
        return [t.clone() for t in (self.theta, self.adam_m, self.adam_v, self.step_dev)]

    def restore(self, snap):
        for t, s in zip((self.theta, self.adam_m, self.adam_v, self.step_dev), snap):
            t.copy_(s)
        self.step_count = int(self.step_dev.item())

    def _bcast_ell(self, lam_row, n):
        return lam_row.reshape(-1, 1).expand(self.d, n).contiguous()

    def _kernel_fwd(self, x1, f1, x2, f2, scale, u=None, out=None):
        if self.variant == "diag":
            return self.o.gibbs_diag_fwd(x1, f1, x2, f2, scale, u=u, out=out)
        return self.o.gibbs_full_fwd(x1, f1, x2, f2, self.kernel_jitter, scale, u=u, out=out)

    def _kernel_bwd(self, x1, f1, x2, f2, scale, **kw):
        if self.variant == "diag":
            r = self.o.gibbs_diag_bwd(x1, f1, x2, f2, scale, **kw)
            return r["d_ell1"], r["d_ell2"], r["d_x1"], r["d_x2"], r["d_scale"]
        r = self.o.gibbs_full_bwd(x1, f1, x2, f2, self.kernel_jitter, scale, **kw)
        return r["d_S1"], r["d_S2"], r["d_x1"], r["d_x2"], r["d_scale"]

    def _solve_spd(self, P, rhs):
        """K^-1 rhs with K = L L^T, P = L^-1.  rhs (M,) or (M,k)."""
        o = self.o
        if rhs.dim() == 1:
            return o.colwsum(P, w=o.gemv_n(P, rhs))
        k = rhs.shape[1]
        kp = max(2, (k + 1) // 2 * 2)
        R = torch.zeros(self.M, kp, dtype=torch.float64, device=self.dev)
        R[:, :k] = rhs
        T = o.dgemm(P, R, tri_a=1)
        return o.dgemm(P, T, transA=True, tri_a=2)[:, :k].contiguous()

    # ------------------------------------------------------------------------------------------------------------------
    def _field_z(self):
        """Latent field at the inducing points: ell_z (D,M) or packed Sigma_z (M,P)."""
        if self.variant == "diag":
            return torch.exp(self.p["log_ell_z"])
        return self.o.sigma_from_h_fwd(self.p["H"], self.p["D"])

    def _rowquad(self, K, C, T=None):
        return self.o.rowquad(K, C, T=T)

    # ---- int8 tensor-core path: K(X_B, Z) exists only as byte-digit planes (csrc/gibbs_digits.cu, csrc/oz8.cu) -------
    def _digits_mode(self):
        return self.rowquad_impl == "i8" and self.M % 128 == 0 and hasattr(self.o, "o8_rowquad_digits")

    def _digit_buffers(self, n):
        """Persistent scratch for a local batch of n rows: digit planes of K and C, the T matrix, the deterministic partial
        buffers.  Created on first use (before graph capture: capture() warms the step up first)."""
        w = self._i8_bufs.get(n)
        if w is None:
            o, M, dev = self.o, self.M, self.dev
            f64 = dict(dtype=torch.float64, device=dev)
            u8 = dict(dtype=torch.uint8, device=dev)
            nsplit = o.gibbs_digits_splits(n, M)
            w = self._i8_bufs[n] = dict(
                Ad=torch.empty(o.digits_bytes(n, M, 128), **u8), Cd=torch.empty(o.digits_bytes(M, M, 64), **u8),
                cexp=torch.empty(M, dtype=torch.int32, device=dev), T=torch.empty(n, M, **f64),
                mu_part=torch.empty(nsplit, n, **f64), q_part=torch.empty(M // 64, n, **f64),
                du_part=torch.empty((n + 127) // 128, M, **f64),
                syrk_part=torch.empty(max(1, o.o8_syrk_part_bytes(n, M) // 8), **f64),
                skip_count=torch.zeros(1, dtype=torch.int32, device=dev),
                skip_rows=torch.empty(n, dtype=torch.int32, device=dev))
        return w

    def _kernel_fwd_digits(self, x1, f1, x2, f2, scale, u, w):
        if self.variant == "diag":
            self.o.gibbs_diag_fwd_digits(x1, f1, x2, f2, scale, w["Ad"], u=u, Ku_part=w["mu_part"])
        else:
            self.o.gibbs_full_fwd_digits(x1, f1, x2, f2, self.kernel_jitter, scale, w["Ad"], u=u, Ku_part=w["mu_part"])

    def _note(self, info=None, loss=None):
        """Record a failed factorisation / non-finite loss in the sticky device flag (no host synchronisation)."""
        if self.status is not None and hasattr(self.o, "status_update"):
            self.o.status_update(self.status, info, loss)

    def check_status(self) -> int:
        """Host poll of the sticky flag (synchronises): 0 = healthy, bit 0 = Cholesky failure, bit 1 = non-finite loss."""
        return 0 if self.status is None else int(self.status.item())

    def recover(self):
        """After a non-zero status: climb psd_safe_cholesky's jitter ladder (reference models/gibbs_kernels.py:201 through
        GPyTorch: +1e-8, +1e-7, +1e-6 in fp64), clear the flag and drop the captured graph (the jitter is baked into it).
        The failed steps did not touch the parameters (guarded Adam).  Raises once the ladder is exhausted."""
        ladder = [0.0, 1e-8, 1e-7, 1e-6]
        nxt = [j for j in ladder if j > self.extra_jitter]
        if not nxt:
            raise RuntimeError("Kzz not positive definite after adding jitter up to %.1e (status %d)" % (ladder[-1],
                                                                                                      self.check_status()))
        self.extra_jitter = nxt[0]
        self.status.zero_()
        regraph = self._graph is not None
        self._graph = None
        return regraph

    def _fork(self):
        """Run the enclosed launches on the side stream, ordered after everything enqueued so far."""
        if self._side is None or not self.overlap:
            return contextlib.nullcontext()
        self._side.wait_stream(torch.cuda.current_stream())
        return torch.cuda.stream(self._side)

    def _join(self):
        if self._side is not None and self.overlap:
            torch.cuda.current_stream().wait_stream(self._side)

    def _fork2(self):
        """Second side stream, forked from whatever stream is current: for M x M GEMMs that are independent of the
        latency-bound chain running on the current stream (the GEMM fills the SMs the chain leaves idle)."""
        if self._side2 is None or not self.overlap:
            return contextlib.nullcontext()
        self._side2.wait_stream(torch.cuda.current_stream())
        return torch.cuda.stream(self._side2)

    def _join2(self):
        if self._side2 is not None and self.overlap:
            torch.cuda.current_stream().wait_stream(self._side2)

    def _field_prepare(self, fz):
        """Z-side part of the field interpolation (independent of the rows): the prior-kernel factorisations at Z and
        the interpolation weights (alpha for the log-normal field, W = (K_row + 1e-5 I)^-1 H for the matrix field)."""
        o, p, M, d = self.o, self.p, self.M, self.d
        Z = p["Z"]
        c = {}
        if self.variant == "diag":
            alphas, Ps, Ldiag = [], [], []
            for b in range(d):
                lamb = self._bcast_ell(self.prior_lam[b], M)
                Kp = o.gibbs_diag_fwd(Z, lamb, Z, lamb, self.prior_os[b:b + 1])
                Kp.diagonal().add_(1e-4)
                Lb, Pb, info_b = o.potrf_inv(Kp, overwrite=True)
                self._note(info_b)
                alphas.append(self._solve_spd(Pb, p["log_ell_z"][b] - self.prior_c[b]))
                Ps.append(Pb)
                Ldiag.append(torch.diagonal(Lb).clone())
            c.update(alpha=torch.stack(alphas), Ps=Ps, Ldiag=Ldiag, ell_z=fz)
        else:
            lamr = self._bcast_ell(self.row_lam[0], M)
            Kr = o.gibbs_diag_fwd(Z, lamr, Z, lamr, self.row_os)
            Kr.diagonal().add_(1e-5)
            _, Pr, info_r = o.potrf_inv(Kr, overwrite=True)
            self._note(info_r)
            c.update(Pr=Pr, W=self._solve_spd(Pr, p["H"]), lamr=lamr)
        return c

    def _field_apply(self, x, c):
        """Row-side part: the field interpolated to the rows x (matrix free).  Returns fx; adds Hx / ell_x to the cache."""
        o, p = self.o, self.p
        if self.variant == "diag":
            ell_x = o.rbf_matvec_fwd(x, p["Z"], self.prior_lam, self.prior_os, c["alpha"].unsqueeze(-1),
                                     bias=self.prior_c, apply_exp=True).squeeze(-1)
            c["ell_x"] = ell_x
            return ell_x
        Hx = o.rbf_matvec_fwd(x, p["Z"], self.row_lam, self.row_os, c["W"].unsqueeze(0))[0]  # (B,d)
        c["Hx"] = Hx
        return o.sigma_from_h_fwd(Hx, p["D"])

    def _field_forward(self, x, fz=None):
        """Latent field interpolated from Z to the rows x.  Returns (fz, fx, cache)."""
        if fz is None:
            fz = self._field_z()
        c = self._field_prepare(fz)
        return fz, self._field_apply(x, c), c

    def _zz_forward(self, fz, s):
        o, p, M = self.o, self.p, self.M
        Ls = torch.tril(p["Ls"])
        with self._fork2():  # S - I does not depend on the factorisation: under the (latency-bound) Cholesky
            E = o.dgemm(Ls, Ls, transB=True, tri_a=1, tri_b=2) - self.eye
        Kzz = self._kernel_fwd(p["Z"], fz, p["Z"], fz, s)
        Kzz.diagonal().add_(self.jitter_zz + self.extra_jitter)
        L, P, info = o.potrf_inv(Kzz, overwrite=True)
        self._note(info)
        u = o.colwsum(P, w=p["m"])  # P^T m
        self._join2()
        EP = o.dgemm(E, P, tri_b=1)
        C = o.dgemm(P, EP, transA=True, tri_a=2)
        return dict(L=L, P=P, info=info, Ls=Ls, u=u, E=E, EP=EP, C=C)

    # ---- C engine ---------------------------------------------------------------------------------------------------
    def use_c_engine(self, on: bool = True):
        """Route loss_and_grad / train_step through the C-ABI step (needs M % 128 == 0: the digit-plane path)."""
        if on and self.M % 128:
            raise ValueError("the C step needs M % 128 == 0 (got %d)" % self.M)
        self.engine = "c" if on else "python"
        return self

    def _plan(self, Bl, world_size, Bg):
        """npgp_svgp_plan for this batch shape (created on first use: before graph capture, capture() warms up first)."""
        from ._lib import SvgpConfig, check, lib, ptr
        import ctypes as C
        tl = self.timeline.data_ptr() if self.timeline is not None else None
        key = (Bl, world_size, Bg, self.learn_z, self.include_prior, tl)
        ent = self._plans.get(key)
        if ent is not None and ent["extra"] != self.extra_jitter:  # psd_safe_cholesky ladder (recover())
            check(lib().npgp_svgp_set_extra_jitter(ent["handle"], float(self.extra_jitter)), "npgp_svgp_set_extra_jitter")
            ent["extra"] = self.extra_jitter
        if ent is None:
            full = self.variant == "full"
            cfg = SvgpConfig(variant=1 if full else 0, d=self.d, M=self.M, B_local=Bl, N_total=self.N, B_global=Bg,
                             world_size=world_size, jitter_zz=self.jitter_zz, jitter_xx=self.jitter_xx,
                             kernel_jitter=self.kernel_jitter, min_var=1e-6, extra_jitter=self.extra_jitter,
                             learn_z=int(self.learn_z), include_prior=int(self.include_prior),
                             row_os=ptr(self.row_os) if full else None, row_lam=ptr(self.row_lam) if full else None,
                             prior_c=None if full else ptr(self.prior_c), prior_os=None if full else ptr(self.prior_os),
                             prior_lam=None if full else ptr(self.prior_lam), timeline=tl)
            assert lib().npgp_svgp_theta_size(C.byref(cfg)) == self.theta.numel()
            nbytes = lib().npgp_svgp_workspace_bytes(C.byref(cfg))
            ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.dev)
            off = (-ws.data_ptr()) % 256
            handle = C.c_void_p()
            check(lib().npgp_svgp_plan_create(C.byref(handle), C.byref(cfg), ws.data_ptr() + off, nbytes), "npgp_svgp_plan_create")
            ent = self._plans[key] = dict(handle=handle, ws=ws, cfg=cfg, extra=self.extra_jitter)
            if tl is not None:  # the C step stamps its sections into fixed slots
                self._timeline_slots = {name: i for i, name in enumerate(self.c_section_names())}
        return ent

    def _plan_view(self, ent, which, count, dtype=torch.float64):
        """Torch view of one of the plan's workspace buffers (npgp_svgp_buffer)."""
        from ._lib import lib
        addr = lib().npgp_svgp_buffer(ent["handle"], which)
        off = addr - ent["ws"].data_ptr()
        nbytes = count * torch.empty((), dtype=dtype).element_size()
        return ent["ws"][off:off + nbytes].view(dtype)

    def _c_loss_and_grad(self, xb, yb, world_size, B_global):
        from ._lib import check, lib, ptr, stream
        Bl = xb.shape[0]
        Bg = B_global if B_global is not None else Bl * world_size
        ent = self._plan(Bl, world_size, Bg)
        xb, yb = xb.contiguous(), yb.contiguous()
        check(lib().npgp_svgp_elbo_fwd(ent["handle"], ptr(xb), ptr(yb), ptr(self.theta), ptr(self.grad), ptr(self.status),
                                       stream()), "npgp_svgp_elbo_fwd")
        check(lib().npgp_svgp_elbo_bwd(ent["handle"], ptr(xb), ptr(self.theta), ptr(self.grad), stream()), "npgp_svgp_elbo_bwd")
        self.last = dict(info=self._plan_view(ent, 8, 1, torch.int32)[0], mu=self._plan_view(ent, 0, Bl))
        return self.grad[-2]

    def c_section_names(self):
        from ._lib import lib
        return [lib().npgp_svgp_section_name(i).decode() for i in range(lib().npgp_svgp_num_sections())]

    # ------------------------------------------------------------------------------------------------------------------
    def loss_and_grad(self, xb, yb, world_size: int = 1, B_global: Optional[int] = None):
        """Fills self.grad with d(-ELBO)/d(theta) for this rank's rows and returns this rank's share of -ELBO
        (also stored in self.grad[-2]); summing over ranks (one all-reduce of self.grad) gives the global values."""
        if self.engine == "c":
            return self._c_loss_and_grad(xb, yb, world_size, B_global)
        o, p, g, M, d = self.o, self.p, self.g, self.M, self.d
        Z = p["Z"]
        Bl = xb.shape[0]
        Bg = B_global if B_global is not None else Bl * world_size
        rep = 1.0 / world_size  # weight of the replicated (KL / prior) terms on this rank
        s = _softplus(p["raw_outputscale"])
        noise = 1e-4 + _softplus(p["raw_noise"])
        self.grad.zero_()

        fz = self._field_z()
        with self._fork():  # Kzz -> Cholesky -> u, C on the side stream, overlapped with the field interpolation
            with self._sec("zz_fwd(potrf+M^3)"):
                zz = self._zz_forward(fz, s)
        with self._sec("field_fwd"):
            fz, fx, fc = self._field_forward(xb, fz)
        self._join()
        P, u, E, EP, C, Ls = zz["P"], zz["u"], zz["E"], zz["EP"], zz["C"], zz["Ls"]

        # ---- data pass: K(X_B, Z) (+ mean), variance quadratic form, expected log-lik
        digits = self._digits_mode()
        K = q = None
        if digits:
            # K is written once as 7-byte digits and consumed by both tensor-core contractions; every reduction of this
            # branch is two-stage with a fixed order (no FP64 atomics)
            w = self._digit_buffers(Bl)
            with self._sec("kxz_fwd"):
                self._kernel_fwd_digits(xb, fx, Z, fz, s, u, w)
                # d(ELL)/d(mu) does not depend on the variance: K^T g_mu rides on the row-quadratic kernel's K tiles
                mu, gmu_early = o.mu_gmu_parts(yb, w["mu_part"], noise, 1.0 / Bg)
            with self._sec("rowquad"):
                o.o8_slice_rows(C, 64, w["Cd"], w["cexp"])
                T = o.o8_rowquad_digits(Bl, M, w["Ad"], s, w["Cd"], w["cexp"], w["T"], q_part=w["q_part"], gvec=gmu_early,
                                        du_part=w["du_part"])
                du = o.o8_sum_partials(w["du_part"])
            with self._sec("gauss_ell"):
                w["skip_count"].zero_()
                acc, gmu, gv, _ = o.gauss_ell_parts(yb, mu, w["q_part"], s, noise, self.jitter_xx, 1e-6, 1.0 / Bg,
                                                    skip_count=w["skip_count"], skip_rows=w["skip_rows"])
        else:
            with self._sec("kxz_fwd"):
                K, mu = self._kernel_fwd(xb, fx, Z, fz, s, u=u)
            with self._sec("rowquad"):
                T, q = self._rowquad(K, C)
            acc, gmu, gv, _ = o.gauss_ell(yb, mu, q, s, noise, self.jitter_xx, 1e-6, 1.0 / Bg)
        ell = acc[0] / Bg

        # ---- KL and prior (replicated terms)
        sec_kl = self._sec("kl+prior")
        sec_kl.__enter__()
        m = p["m"]
        dLs_diag = torch.diagonal(Ls)
        kl = 0.5 * ((Ls * Ls).sum() + (m * m).sum() - M - torch.log(dLs_diag * dLs_diag).sum())
        lp = torch.zeros((), dtype=torch.float64, device=self.dev)
        if self.include_prior and self.variant == "diag":
            for b in range(d):
                r_b = p["log_ell_z"][b] - self.prior_c[b]
                lp = lp + (-0.5 * (r_b * fc["alpha"][b]).sum() - torch.log(fc["Ldiag"][b]).sum()
                           - 0.5 * M * LOG2PI) / M
        elbo_local = ell + rep * (-kl + lp) / self.N
        sec_kl.__exit__()

        # ---- backward of the data term through K(X_B, Z)
        gv2 = 2.0 * gv
        # Scheduling (all FP64 work shares one pipe, DFMA and DMMA alike): the SYRK runs alone at full rate on the side
        # stream; the latency-bound O(M^3) backward chain that follows it is then hidden under the FP64-bound Gibbs
        # backward on the main stream, which starts when the SYRK has finished.
        # (digit path: the SYRK runs on the int8 tensor pipe and leaves the FP64 pipe, registers and ~50 KB of shared memory
        # per SM free, so the FP64-bound Gibbs backward starts at once and runs beside it)
        wsyrk_done = torch.cuda.Event() if (self._side is not None and self.overlap and not digits) else None
        with self._fork():
            with self._sec("wsyrk"):
                if digits:
                    # every unclamped row has the same weight w0 = acc[3]; clamped rows (normally none) are removed again
                    dC = o.o8_syrk_digits(Bl, M, w["Ad"], s, w["syrk_part"], w0=acc[3:4], skip_count=w["skip_count"],
                                          skip_rows=w["skip_rows"])
                else:
                    du = o.colwsum(K, w=gmu)
                    # gv is constant unless a variance was clamped: acc[2] counts the unclamped rows (decided on the device)
                    dC = o.wsyrk(K, w=gv, uniform_count=acc[2:3], uniform_target=float(Bl))
            if wsyrk_done is not None:
                wsyrk_done.record()
            with self._sec("m3_bwd+kzz_bwd"):
                dm = o.gemv_n(P, du)
                # dE = P dC P^T and E dE = (E P)(dC P^T): with W = dC P^T both follow from ONE product, so the chain to dKzz is
                # W -> X -> P^T X -> (P^T X) P (four dependent GEMMs instead of five); dE itself only feeds the dL_s branch
                W = o.dgemm(dC, P, transB=True, tri_b=2)
                with self._fork2():  # dL_s branch, independent of the dKzz chain below
                    dE = o.dgemm(P, W, tri_a=1)
                    dLs = torch.tril(o.dgemm(dE, Ls, alpha=2.0, tri_b=1))
                    g["m"].copy_(-(dm - rep * m / self.N))
                    g["Ls"].copy_(-(dLs - rep * (Ls - torch.diag(1.0 / dLs_diag)) / self.N))
                X = o.dgemm(EP, W, alpha=2.0)
                X.addr_(m, dm)
                o.phi_mask_(X, -1.0)
                dK = o.dgemm(o.dgemm(P, X, transA=True, tri_a=2, tri_b=1), P, tri_b=1)
                dKzz = 0.5 * (dK + dK.T)
                dfz1, dfz2, dZ1, dZ2, ds2 = self._kernel_bwd(Z, fz, Z, fz, s, G=dKzz, need_dx1=self.learn_z,
                                                             need_dx2=self.learn_z, need_dscale=True)
                self._join2()
        if wsyrk_done is not None:
            torch.cuda.current_stream().wait_event(wsyrk_done)
        with self._sec("kxz_bwd"):
            dfx, dfz, _, dZ, ds = self._kernel_bwd(xb, fx, Z, fz, s, G=T, rowscale=gv2, rowvec=gmu, colvec=u,
                                                   need_dx2=self.learn_z, need_dscale=True)
        ds = ds + gv.sum()  # v = s + ...

        # ---- backward through the field interpolation: the row-side part needs only dfx (main stream, before the join)
        sec_f = self._sec("field_bwd")
        sec_f.__enter__()
        gZ = torch.zeros_like(Z)
        if self.variant == "diag":
            alpha, ell_x, ell_z = fc["alpha"], fc["ell_x"], fc["ell_z"]
            dlog = (dfx * ell_x).unsqueeze(-1)
            dalpha, dZf = o.rbf_matvec_bwd(xb, Z, self.prior_lam, self.prior_os, alpha.unsqueeze(-1), dlog,
                                           need_dz=self.learn_z)
            g_logell = torch.zeros_like(ell_z)
            for b in range(d):
                Pb = fc["Ps"][b]
                beta = self._solve_spd(Pb, dalpha[b, :, 0])
                g_logell[b] += beta
                pw = rep / (self.N * M) if self.include_prior else 0.0
                if self.include_prior:
                    g_logell[b] -= pw * alpha[b]
                if self.learn_z:
                    lamb = self._bcast_ell(self.prior_lam[b], M)
                    # dELBO/dKp_b = -beta alpha^T  (+ prior: pw (0.5 alpha alpha^T - 0.5 Kp^-1))
                    Gm = None
                    rv, cv = -beta, alpha[b]
                    if self.include_prior:
                        Gm = o.dgemm(Pb, Pb, transA=True, alpha=-0.5 * pw, tri_a=2, tri_b=1)
                        rv = rv + 0.5 * pw * alpha[b]
                    r = o.gibbs_diag_bwd(Z, lamb, Z, lamb, self.prior_os[b:b + 1], G=Gm, rowvec=rv, colvec=cv,
                                         need_dx1=True, need_dx2=True)
                    gZ += r["d_x1"] + r["d_x2"]
            if self.learn_z:
                gZ += dZf
        else:
            dHx, dD1 = o.sigma_from_h_bwd(fc["Hx"], p["D"], dfx)
            dW, dZf = o.rbf_matvec_bwd(xb, Z, self.row_lam, self.row_os, fc["W"].unsqueeze(0), dHx.unsqueeze(0),
                                       need_dz=self.learn_z)
            beta = self._solve_spd(fc["Pr"], dW[0])  # (M,d) = Kr^-1 dW
            if self.learn_z:
                kp = 4
                b4 = torch.zeros(M, kp, dtype=torch.float64, device=self.dev)
                w4 = torch.zeros(M, kp, dtype=torch.float64, device=self.dev)
                b4[:, :d], w4[:, :d] = beta, fc["W"]
                Gk = o.dgemm(b4, w4, transB=True, alpha=-1.0)  # dELBO/dKr = -beta W^T
                r = o.gibbs_diag_bwd(Z, fc["lamr"], Z, fc["lamr"], self.row_os, G=Gk, need_dx1=True, need_dx2=True)
                gZ += dZf + r["d_x1"] + r["d_x2"]
        sec_f.__exit__()

        # ---- join the O(M^3) chain and assemble the flat gradient
        self._join()
        sec_m3 = self._sec("assemble")
        sec_m3.__enter__()
        dfz = dfz + dfz1 + dfz2
        ds = ds + ds2
        if self.learn_z:
            gZ += dZ + dZ1 + dZ2
        if self.variant == "diag":
            g["log_ell_z"].copy_(-(g_logell + dfz * ell_z))
        else:
            dHz, dD2 = o.sigma_from_h_bwd(p["H"], p["D"], dfz)
            g["H"].copy_(-(beta + dHz))
            g["D"].copy_(-(dD1 + dD2))
        g["Z"].copy_(-gZ)
        g["raw_outputscale"].copy_(-(ds * torch.sigmoid(p["raw_outputscale"])).reshape(1))
        dnoise = (0.5 / Bg) * (acc[1] / (noise * noise) - Bl / noise)
        g["raw_noise"].copy_(-(dnoise * torch.sigmoid(p["raw_noise"])).reshape(1))
        self.grad[-2] = -elbo_local.reshape(())
        sec_m3.__exit__()
        self.last = dict(info=zz["info"], ell=ell, kl=kl, log_prior=lp, mu=mu)
        return self.grad[-2]

    # ------------------------------------------------------------------------------------------------------------------
    def adam_step(self, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8):
        self.step_count += 1
        g = self.grad[:self.theta.numel()]
        if self.status is not None and hasattr(self.o, "adam_step_guarded_"):
            # the (all-reduced, hence rank-consistent) loss is checked here: a NaN on any rank stops the update on all
            self._note(None, self.grad[-2:-1])
            # step counter on the device (identical eagerly and under graph replay); no update while the status flag is set
            self.o.adam_step_guarded_(self.theta, g, self.adam_m, self.adam_v, self.step_dev, self.status, lr, beta1, beta2, eps,
                                      1.0, self.mask)
        elif hasattr(self.o, "adam_step_dev_"):
            self.o.adam_step_dev_(self.theta, g, self.adam_m, self.adam_v, self.step_dev, lr, beta1, beta2, eps, 1.0,
                                  self.mask)
        else:
            self.o.adam_step_(self.theta, g, self.adam_m, self.adam_v, self.step_count, lr, beta1, beta2, eps, 1.0,
                              self.mask)

    def train_step(self, xb, yb, lr=0.01, world_size=1, B_global=None, all_reduce=None):
        """loss_and_grad -> (all-reduce of the flat gradient) -> Adam.  Returns the (global) loss as a device scalar."""
        from .comm import NpgpComm
        if self.engine == "c" and (isinstance(all_reduce, NpgpComm) or (all_reduce is None and world_size == 1)):
            # the whole step is ONE C call (npgp_svgp_step): forward, backward, all-reduce on the npgp communicator, guarded Adam
            from ._lib import check, lib, ptr, stream
            Bl = xb.shape[0]
            ent = self._plan(Bl, world_size, B_global if B_global is not None else Bl * world_size)
            xb, yb = xb.contiguous(), yb.contiguous()
            check(lib().npgp_svgp_step(ent["handle"], ptr(xb), ptr(yb), ptr(self.theta), ptr(self.grad), ptr(self.adam_m),
                                       ptr(self.adam_v), ptr(self.mask), ptr(self.step_dev), ptr(self.status), float(lr), 0.9,
                                       0.999, 1e-8, all_reduce.handle if all_reduce is not None else None, stream()),
                  "npgp_svgp_step")
            self.step_count += 1
            return self.grad[-2]
        self.loss_and_grad(xb, yb, world_size, B_global)
        if all_reduce is not None:
            with self._sec("allreduce"):
                all_reduce(self.grad)
        with self._sec("adam"):
            self.adam_step(lr)
        return self.grad[-2]

    # ---- CUDA-graph execution: the ~250 launches of a step are captured once and replayed ---------------------------
    def capture(self, B_local: int, world_size: int = 1, B_global: Optional[int] = None, lr: float = 0.01, all_reduce=None,
                buffers: int = 1):
        """Capture the whole step for minibatches of B_local rows: loss_and_grad, the all-reduce of the flat gradient
        (`all_reduce(self.grad)`, e.g. an NCCL all-reduce -- NCCL collectives are capturable) and the Adam update, so a
        replay is one graph launch on every rank.  Without `all_reduce` and world_size > 1 the collective and Adam run
        after the replayed graph (train_step_graph(all_reduce=...)).
        buffers = 2: two graphs over two static input buffers, used alternately, so that the host-to-device copy of the next
        minibatch (on a copy stream) runs under the current step (train_step_graph_async / loss_result)."""
        f64 = dict(dtype=torch.float64, device=self.dev)
        self._gxs = [torch.zeros(B_local, self.d, **f64) for _ in range(buffers)]
        self._gys = [torch.zeros(B_local, **f64) for _ in range(buffers)]
        self._gx, self._gy = self._gxs[0], self._gys[0]
        self._g_world, self._g_lr = world_size, lr
        self._g_fused = world_size == 1 or all_reduce is not None
        snap = [t.clone() for t in (self.theta, self.adam_m, self.adam_v, self.step_dev)]
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream())
        c_fused = self.engine == "c" and self._g_fused
        with torch.cuda.stream(side):  # warm-up off the default stream (allocator pools, lazy attribute calls)
            for _ in range(2):
                if c_fused:
                    self.train_step(self._gx, self._gy, lr, world_size, B_global, all_reduce)
                    continue
                self.loss_and_grad(self._gx, self._gy, world_size, B_global)
                if all_reduce is not None:
                    all_reduce(self.grad)  # communicator set-up must not happen under capture
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._graphs = []
        for gx, gy in zip(self._gxs, self._gys):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                if c_fused:
                    self.train_step(gx, gy, lr, world_size, B_global, all_reduce)
                else:
                    self.loss_and_grad(gx, gy, world_size, B_global)
                    if self._g_fused:
                        if all_reduce is not None:
                            all_reduce(self.grad)
                        self.adam_step(lr)
            self._graphs.append(graph)
        self._graph = self._graphs[0]
        # (the graphs hold raw pointers into the plan workspace / self._i8_bufs, which live as long as the model)
        for t, s in zip((self.theta, self.adam_m, self.adam_v, self.step_dev), snap):
            t.copy_(s)
        self.step_count = int(self.step_dev.item())
        # pipelined replay (train_step_graph_async): copy stream, per-buffer events, pinned slots for the loss
        self._g_next = 0
        self._copy_stream = torch.cuda.Stream(device=self.dev)
        self._g_done = [torch.cuda.Event() for _ in range(buffers)]
        self._g_copied = [torch.cuda.Event() for _ in range(buffers)]
        self._loss_ev = [torch.cuda.Event() for _ in range(buffers)]
        self._loss_host = torch.zeros(buffers, dtype=torch.float64).pin_memory()
        for e in self._g_done:
            e.record()

    def train_step_graph(self, xb, yb, all_reduce=None):
        """Replay of the captured step on a new minibatch (xb, yb may live in pinned host memory)."""
        self._gx.copy_(xb, non_blocking=True)
        self._gy.copy_(yb, non_blocking=True)
        self._graph.replay()
        if not self._g_fused:
            if all_reduce is not None:
                all_reduce(self.grad)
            self.adam_step(self._g_lr)
        else:
            self.step_count += 1
        return self.grad[-2]

    def train_step_graph_async(self, xb, yb):
        """Pipelined replay (needs capture(..., buffers >= 2) and a fused graph): the minibatch is copied into the next static
        input buffer on the copy stream -- ordered only after the step that last READ that buffer, so it runs under the step
        in flight --, the step is replayed, and its loss is copied to a pinned host slot asynchronously.  Returns a ticket
        for loss_result(); call that for step k after enqueuing step k + 1 and the host never stalls the device."""
        assert self._g_fused and len(self._graphs) >= 2, "capture(..., buffers=2) with the collective inside the graph"
        i = self._g_next
        cur = torch.cuda.current_stream()
        self._copy_stream.wait_event(self._g_done[i])
        with torch.cuda.stream(self._copy_stream):
            self._gxs[i].copy_(xb, non_blocking=True)
            self._gys[i].copy_(yb, non_blocking=True)
            self._g_copied[i].record(self._copy_stream)
        cur.wait_event(self._g_copied[i])
        self._graphs[i].replay()
        self._g_done[i].record(cur)
        self._loss_host[i:i + 1].copy_(self.grad[-2:-1], non_blocking=True)
        self._loss_ev[i].record(cur)
        self.step_count += 1
        self._g_next = (i + 1) % len(self._graphs)
        return i

    def loss_result(self, ticket: int) -> float:
        """The (global) loss of the step train_step_graph_async returned `ticket` for (waits for that step only)."""
        self._loss_ev[ticket].synchronize()
        return float(self._loss_host[ticket])

    @torch.no_grad()
    def predict(self, xs, chunk: int = 1 << 18):
        """Posterior marginal mean and variance of f at xs (rows can be sharded across ranks by the caller; no
        collective is involved).  Z-side factors are computed once, rows are streamed in chunks."""
        o, p = self.o, self.p
        s = _softplus(p["raw_outputscale"])
        fz = self._field_z()
        fc = self._field_prepare(fz)
        zz = self._zz_forward(fz, s)
        n = xs.shape[0]
        mean = torch.empty(n, dtype=torch.float64, device=self.dev)
        var = torch.empty(n, dtype=torch.float64, device=self.dev)
        K = T = None
        digits = self._digits_mode()
        if digits:
            w0 = self._digit_buffers(min(chunk, n))
            o.o8_slice_rows(zz["C"], 64, w0["Cd"], w0["cexp"])
        for lo in range(0, n, chunk):
            xc = xs[lo:lo + chunk].contiguous()
            fx = self._field_apply(xc, fc)
            nc = xc.shape[0]
            if digits:
                w = self._digit_buffers(nc)
                self._kernel_fwd_digits(xc, fx, p["Z"], fz, s, zz["u"], w)
                o.o8_rowquad_digits(nc, self.M, w["Ad"], s, w0["Cd"], w0["cexp"], w["T"], q_part=w["q_part"])
                mu, q = w["mu_part"].sum(0), w["q_part"].sum(0)
            else:
                if K is None or K.shape[0] != nc:
                    K = torch.empty(nc, self.M, dtype=torch.float64, device=self.dev)
                    T = torch.empty_like(K)
                _, mu = self._kernel_fwd(xc, fx, p["Z"], fz, s, u=zz["u"], out=K)
                _, q = self._rowquad(K, zz["C"], T=T)
            mean[lo:lo + chunk] = mu
            var[lo:lo + chunk] = (s + self.jitter_xx + q).clamp_min(1e-6)
        return mean, var

    @torch.no_grad()
    def predictive(self, xs, y=None, *, field: bool = False, chunk: int = 65536) -> Predictive:
        """Posterior marginals at xs through the C ABI (npgp_svgp_predict_prepare + npgp_svgp_predict): one call for the
        Z-side factors, one for all rows, streamed in chunks of `chunk` rows through the plan of a single-rank C-engine run
        with that batch size (no allocation per chunk; the row-side reductions have a fixed order).  Works whichever engine
        trains the model; same arithmetic as predict().  Needs M % 128 == 0 (the digit-plane path)."""
        if self.M % 128:
            raise ValueError("the C prediction needs M % 128 == 0 (got %d)" % self.M)
        from ._lib import check, lib, ptr, stream
        ent = self._plan(chunk, 1, chunk)
        xs = xs.contiguous()
        n = xs.shape[0]
        f64 = dict(dtype=torch.float64, device=self.dev)
        mean, var, var_y = (torch.empty(n, **f64) for _ in range(3))
        fld = lpd = sums = None
        if field:
            fld = torch.empty(self.d, n, **f64) if self.variant == "diag" else torch.empty(n, self.d * (self.d + 1) // 2, **f64)
        if y is not None:
            y = y.contiguous()
            lpd, sums = torch.empty(n, **f64), torch.zeros(3, **f64)
        check(lib().npgp_svgp_predict_prepare(ent["handle"], ptr(self.theta), ptr(self.status), stream()),
              "npgp_svgp_predict_prepare")
        check(lib().npgp_svgp_predict(ent["handle"], n, ptr(xs), ptr(y), ptr(self.theta), ptr(mean), ptr(var), ptr(var_y),
                                      ptr(fld), ptr(lpd), ptr(sums), stream()), "npgp_svgp_predict")
        return Predictive(mean, var, var_y, fld, lpd, sums)

    @torch.no_grad()
    def sample(self, xs, num_samples: int, *, seed: int = 0, noise: bool = False, row_offset: int = 0,
               chunk: int = 65536) -> torch.Tensor:
        """num_samples posterior draws of f (noise=True: of y) at xs, correlated across rows: (num_samples, n).  Goes through
        the C ABI (npgp_svgp_predict_prepare, npgp_svgp_sample_prepare, npgp_svgp_sample) on the same plan as predictive();
        the mean of the draws is predictive().mean.  Draw s at global row row_offset + i depends only on seed, s and that row,
        so rows sharded over ranks with their global offsets are parts of one joint draw.  The draws are the modified
        predictive process under q(u) (see npgp_svgp_sample in include/npgp.h).  Needs M % 128 == 0 (the digit-plane path)."""
        if self.M % 128:
            raise ValueError("the C sampler needs M % 128 == 0 (got %d)" % self.M)
        from ._lib import check, lib, ptr, stream
        import ctypes as C
        ent = self._plan(chunk, 1, chunk)
        xs = xs.contiguous()
        n = xs.shape[0]
        nbytes = lib().npgp_svgp_sample_workspace_bytes(C.byref(ent["cfg"]), int(num_samples))
        if nbytes < 0:
            raise ValueError("num_samples must be in 1 .. 1024 (got %d)" % num_samples)
        work = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.dev)
        wp = work.data_ptr() + (-work.data_ptr()) % 256
        out = torch.empty(int(num_samples), n, dtype=torch.float64, device=self.dev)
        check(lib().npgp_svgp_predict_prepare(ent["handle"], ptr(self.theta), ptr(self.status), stream()),
              "npgp_svgp_predict_prepare")
        check(lib().npgp_svgp_sample_prepare(ent["handle"], ptr(self.theta), int(num_samples), int(seed), wp, nbytes, stream()),
              "npgp_svgp_sample_prepare")
        check(lib().npgp_svgp_sample(ent["handle"], n, ptr(xs), int(row_offset), ptr(self.theta), int(bool(noise)), ptr(out),
                                     n, wp, nbytes, stream()), "npgp_svgp_sample")
        return out
