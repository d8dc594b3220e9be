"""Matrix-free (streamed) SGPR objective for the diagonal Gibbs kernel: the collapsed bound of DiagonalSparseGP
(reference models/nonstationary_models.py:64-89 driving models/gibbs_kernels.py:187-261; SURVEY.md 3.2 / Appendix A.6)
evaluated WITHOUT materialising the N x M root, so that it runs at the scale of BASELINE config 3 (N = 4M rows,
M = 2048), where the reference's `k_ux1.matmul(inv_root)` would need 68 GB.

With K = Gibbs(X, Z) (unscaled, rows streamed in chunks) and the root rows G = K L^-T (Kzz = L L^T) the bound depends on
the rows only through
    W = G^T G (M x M SYRK),   c = G^T y,   y^T y,
so one pass over the rows accumulates just those (each chunk is whitened by a triangular GEMM first: accumulating the
unwhitened K^T K is cheaper but numerically unusable at N ~ 1e6, see neg_objective_and_grad).  Everything else is M x M
algebra on the blocked Cholesky / GEMM kernels (differentiated by the autograd Functions of `functional.py`).  The
data-side gradient needs a second pass: dObj/dG_chunk = G_chunk (dW + dW^T) + y_chunk dc^T, pushed back through the
whitening (dK = dG L^-1, dL^-1 += dG^T K) and consumed inside the analytic Gibbs backward kernel (never stored as a
gradient matrix); the lengthscale field is interpolated matrix free in both passes.  Rows shard over ranks: W, c, y^T y
and the gradients are sums.  The large products run on the int8 tensor cores (exact Ozaki split, csrc/ozaki.cu) when M
is a multiple of 128, on the FP64 tensor pipe otherwise."""
from __future__ import annotations

import math
from typing import Optional

import torch

from . import functional as F
from . import ops

LOG2PI = math.log(2.0 * math.pi)


def _softplus(x):
    return torch.nn.functional.softplus(x)


def _syrk(Fc, out, use_i8=True):
    """F^T F of a chunk: exact int8 tensor-core path when the width allows (multiple of 128), else FP64 DMMA."""
    if use_i8 and Fc.shape[1] % 128 == 0 and Fc.is_contiguous():
        return ops.syrk_i8(Fc, out=out)
    return ops.wsyrk(Fc, out=out)


def _rowmul(Fc, Csym, T, use_i8=True):
    """T = F_chunk @ Csym (Csym symmetric) on the int8 tensor cores when the width allows (multiple of 64)."""
    if use_i8 and Fc.shape[1] % 64 == 0 and Fc.is_contiguous():
        return ops.rowquad_i8(Fc, Csym, need_q=False, T=T)
    return ops.rowquad(Fc, Csym, need_q=False, T=T)


def _inv_softplus(v: float) -> float:
    return v + math.log(-math.expm1(-v))


class SGPRGibbsStream(torch.nn.Module):
    def __init__(self, Z, log_ell_z, prior_c, prior_os, prior_lam, outputscale=0.644, noise=0.011,
                 learn_inducing_locations=True, include_prior=True, jitter_zz=0.0):
        super().__init__()
        self.jitter_zz = jitter_zz
        self.Z = torch.nn.Parameter(Z.clone(), requires_grad=learn_inducing_locations)
        self.log_ell_z = torch.nn.Parameter(log_ell_z.clone())
        self.raw_outputscale = torch.nn.Parameter(torch.tensor([_inv_softplus(outputscale)], dtype=torch.float64,
                                                               device=Z.device))
        self.raw_noise = torch.nn.Parameter(torch.tensor([_inv_softplus(noise - 1e-4)], dtype=torch.float64,
                                                         device=Z.device))
        self.register_buffer("prior_c", prior_c.clone())
        self.register_buffer("prior_os", prior_os.clone())
        self.register_buffer("prior_lam", prior_lam.clone())
        self.include_prior = include_prior

    # ------------------------------------------------------------------------------------------------------------------
    def _z_side(self):
        """Autograd graph of everything that depends on Z-side parameters only."""
        M, D = self.Z.shape
        ell_z = torch.exp(self.log_ell_z)
        eye = torch.eye(M, dtype=torch.float64, device=self.Z.device)
        alphas, lp = [], self.Z.new_zeros(())
        for b in range(D):
            Kp = F.rbf_ard(self.Z, self.Z, self.prior_lam[b], self.prior_os[b]) + 1e-4 * eye
            Lb, Pb = F.psd_safe_chol_inv(Kp)
            r = self.log_ell_z[b] - self.prior_c[b]
            a = F.spd_solve(Pb, r)
            alphas.append(a)
            if self.include_prior:  # LogNormalPriorProcess.log_prob (gibbs_kernels.py:102-109): per dim, divided by M
                lp = lp + (-0.5 * (r * a).sum() - torch.log(torch.diagonal(Lb)).sum() - 0.5 * M * LOG2PI) / M
        alpha = torch.stack(alphas)
        Kzz = F.gibbs_diag(self.Z, ell_z, self.Z, ell_z)
        # psd_safe_cholesky ladder (gibbs_kernels.py:201), keeping the jittered matrix: it is reused in Sigma below
        for jit in (0.0, 1e-8, 1e-7, 1e-6):
            Kj = Kzz + (self.jitter_zz + jit) * eye
            L, P, info = F.chol_inv(Kj)
            if int(info) == 0:
                break
        else:
            raise RuntimeError("Kzz not positive definite after adding jitter up to 1e-6")
        return ell_z, alpha, (Kj, L, P), lp

    def _chunk_forward(self, xc, ell_z, alpha, K_out=None):
        ell_x = ops.rbf_matvec_fwd(xc, self.Z.detach(), self.prior_lam, self.prior_os, alpha.unsqueeze(-1),
                                   bias=self.prior_c, apply_exp=True).squeeze(-1)
        K = ops.gibbs_diag_fwd(xc, ell_x, self.Z.detach(), ell_z, out=K_out)
        return ell_x, K

    def _pass1(self, x, y, chunk, ell_zd, alphad, Pd, all_reduce):
        """Pass 1 over this rank's rows: W = G^T G, c = G^T y, y^T y of the whitened root rows G = K P^T, summed over ranks by
        `all_reduce`.  Also returns the chunk buffers (K, G) for the caller's second pass."""
        dev = x.device
        n_loc = x.shape[0]
        M = self.Z.shape[0]
        use_i8 = getattr(self, "use_i8", True)
        W = torch.zeros(M, M, dtype=torch.float64, device=dev)
        c = torch.zeros(M, dtype=torch.float64, device=dev)
        yy = torch.zeros((), dtype=torch.float64, device=dev)
        rows = min(chunk, n_loc)
        Kbuf = torch.empty(rows, M, dtype=torch.float64, device=dev)
        Gbuf = torch.empty_like(Kbuf)
        Wc = torch.empty_like(W)
        for lo in range(0, n_loc, chunk):
            xc, yc = x[lo:lo + chunk].contiguous(), y[lo:lo + chunk].contiguous()
            _, K = self._chunk_forward(xc, ell_zd, alphad, Kbuf[:xc.shape[0]])
            G = ops.dgemm(K, Pd, transB=True, tri_b=2, C=Gbuf[:xc.shape[0]])
            W += _syrk(G, Wc, use_i8)
            ops.colwsum(G, w=yc, out=c)
            yy += (yc * yc).sum()
        if all_reduce is not None:
            packed = torch.cat([W.reshape(-1), c, yy.reshape(1)])
            all_reduce(packed)
            W, c, yy = packed[:M * M].reshape(M, M), packed[M * M:M * M + M], packed[-1]
        return W, c, yy, Kbuf, Gbuf

    @torch.no_grad()
    def posterior(self, x, y, *, chunk: int = 65536, n_total: Optional[int] = None, all_reduce=None) -> "SGPRPosterior":
        """The collapsed SGPR posterior at the current parameters, from one pass over this rank's training rows (x, y) --
        the pass 1 of neg_objective_and_grad, all-reduced the same way.  Returns a snapshot: later parameter updates do not
        change it.  With B = I + (s/noise) W and P_B = chol(B)^-1, a test row with whitened features g = P k(x) has
            mean = (s/noise) g^T B^-1 c = k^T u,    var_f = s max(1 - |P k|^2, 0) + |V k|^2,    V = sqrt(s) P_B P,
        the second term being the reference's eval-time diagonal correction (gibbs_kernels.py:228-232).  `n_total` is
        accepted for symmetry with neg_objective_and_grad; the posterior does not depend on it."""
        del n_total
        ell_z, alpha, (_, _, P), _ = self._z_side()
        ell_z, alpha, P = ell_z.contiguous(), alpha.contiguous(), P.contiguous()
        W, c, _, _, _ = self._pass1(x, y, chunk, ell_z, alpha, P, all_reduce)
        M = self.Z.shape[0]
        s = _softplus(self.raw_outputscale).reshape(())
        noise = (1e-4 + _softplus(self.raw_noise)).reshape(())
        Bm = torch.eye(M, dtype=torch.float64, device=x.device) + (s / noise) * (0.5 * (W + W.T))
        _, PB = F.psd_safe_chol_inv(Bm)
        u = F.matmul(P.T, F.matmul(PB.T, F.matmul(PB, c))) * (s / noise)
        V = ops.dgemm(F._aligned(PB), F._aligned(P), tri_a=1, tri_b=1, out_tri=1, C=torch.zeros_like(P))
        V *= torch.sqrt(s)
        return SGPRPosterior(self, "diag", P=P, V=V, u=u, s=s, noise=noise, ell_z=ell_z, alpha=alpha,
                             use_i8=getattr(self, "use_i8", True))

    def neg_objective_and_grad(self, x, y, chunk: int = 65536, n_total: Optional[int] = None, all_reduce=None,
                               world_size: int = 1):
        """Fills .grad of the parameters with the gradient of MINUS the collapsed SGPR objective (divided by n, as
        ExactMarginalLogLikelihood does) and returns its value.  `x`, `y`: this rank's rows; `n_total`: global row count;
        `all_reduce(t)` sums a tensor over ranks (W, c, y^T y after pass 1; the data-side gradients after pass 2).

        Rows are whitened chunk by chunk before they are accumulated, G = K L^-T (the reference's own root,
        gibbs_kernels.py:225), so that B = I + (s/noise) G^T G has eigenvalues >= 1 and log det Kzz cancels: accumulating
        the unwhitened Gram matrix K^T K instead (12 instead of 22 M^2 flop per row) was measured to move the objective by
        4e-5 at N = 4.2e6 when K^T K changed in its last bits -- `Kzz + (s/noise) K^T K` is too ill-conditioned there."""
        dev = x.device
        n_loc = x.shape[0]
        n = n_total if n_total is not None else n_loc
        M, D = self.Z.shape
        use_i8 = getattr(self, "use_i8", True)
        ell_z, alpha, (_, _, P), lp = self._z_side()
        ell_zd, alphad, Pd = ell_z.detach().contiguous(), alpha.detach().contiguous(), P.detach()

        W, c, yy, Kbuf, Gbuf = self._pass1(x, y, chunk, ell_zd, alphad, Pd, all_reduce)
        W = W.clone().requires_grad_(True)
        c = c.clone().requires_grad_(True)

        # ---- M x M algebra: B = I + (s/noise) W
        s = _softplus(self.raw_outputscale).reshape(())
        noise = (1e-4 + _softplus(self.raw_noise)).reshape(())
        Bm = torch.eye(M, dtype=torch.float64, device=dev) + (s / noise) * (0.5 * (W + W.T))
        LB, PB = F.psd_safe_chol_inv(Bm)
        w = F.matmul(PB, c)
        quad = yy / noise - (s / (noise * noise)) * (w * w).sum()
        logdet = 2.0 * torch.log(torch.diagonal(LB)).sum() + n * torch.log(noise)
        ll = -0.5 * (quad + logdet + n * LOG2PI)
        trace = -0.5 * (n - torch.diagonal(W).sum()) / noise  # unscaled kernel (gibbs_kernels.py:256-260)
        obj = (ll + trace + lp) / n
        loss = -obj
        dW, dc = torch.autograd.grad(loss, [W, c], retain_graph=True)
        dW2 = (dW + dW.T).contiguous()
        dc = dc.contiguous()

        # ---- pass 2: dG = G (dW + dW^T) + y dc^T;  dK = dG P (to the analytic Gibbs backward);  dP += dG^T K
        d_ell_z = torch.zeros_like(ell_zd)
        dZ = torch.zeros_like(self.Z)
        dalpha = torch.zeros(D, M, 1, dtype=torch.float64, device=dev)
        dP = torch.zeros(M, M, dtype=torch.float64, device=dev)
        Tbuf = torch.empty_like(Kbuf)
        need_dz = self.Z.requires_grad
        for lo in range(0, n_loc, chunk):
            xc, yc = x[lo:lo + chunk].contiguous(), y[lo:lo + chunk].contiguous()
            ell_x, K = self._chunk_forward(xc, ell_zd, alphad, Kbuf[:xc.shape[0]])
            G = ops.dgemm(K, Pd, transB=True, tri_b=2, C=Gbuf[:xc.shape[0]])
            T, _ = _rowmul(G, dW2, Tbuf[:xc.shape[0]], use_i8)
            T.addcmul_(yc.unsqueeze(1), dc.unsqueeze(0))
            ops.dgemm(T, K, transA=True, beta=1.0, C=dP)
            dK = ops.dgemm(T, Pd, tri_b=1, C=Gbuf[:xc.shape[0]])  # G is no longer needed: reuse its storage
            r = ops.gibbs_diag_bwd(xc, ell_x, self.Z.detach(), ell_zd, None, G=dK, need_dx2=need_dz)
            d_ell_z += r["d_ell2"]
            if need_dz:
                dZ += r["d_x2"]
            dlog = (r["d_ell1"] * ell_x).unsqueeze(-1)
            da, dzf = ops.rbf_matvec_bwd(xc, self.Z.detach(), self.prior_lam, self.prior_os, alphad.unsqueeze(-1), dlog,
                                         need_dz=need_dz)
            dalpha += da
            if need_dz:
                dZ += dzf
        if all_reduce is not None:
            parts = [d_ell_z, dZ, dalpha, dP]
            packed = torch.cat([t.reshape(-1) for t in parts])
            all_reduce(packed)
            out, off = [], 0
            for t in parts:
                out.append(packed[off:off + t.numel()].reshape(t.shape))
                off += t.numel()
            d_ell_z, dZ, dalpha, dP = out

        # ---- finish: Z-side graph (Kzz -> P, prior, alpha) + the streamed contributions
        for p_ in self.parameters():
            p_.grad = None
        torch.autograd.backward([loss, alpha, P], [torch.ones_like(loss), dalpha.squeeze(-1), torch.tril(dP)])
        with torch.no_grad():
            self.log_ell_z.grad += d_ell_z * ell_zd
            if need_dz:
                self.Z.grad += dZ
        return loss.detach()


class SGPRSpatioTemporalStream(torch.nn.Module):
    """Matrix-free collapsed bound of SparseSpatioTemporal_Nonstationary (reference models/spatio_temporal_models.py:35-60
    in training mode, scored by ExactMarginalLogLikelihood): Nystrom (outputscale >= 7)(RBF x Periodic) on time (column 0)
    plus scaled Nystrom Gibbs on (lon, lat) (columns 1, 2), both on ONE inducing set Z (M, 3).  The sum of the two
    Nystrom kernels has the rank-2M root [K_t U_t^-1, sqrt(s) K_s U_s^-1], so the rows enter only through
        A = F^T F (2M x 2M),  b = F^T y,  y^T y,        F = [K_t, K_s]  (n x 2M feature rows, streamed in chunks)
    and the N x 2M root (137 GB at N = 4 194 304, M = 2048) is never formed.  As in the reference the temporal kernel's
    inducing points are a frozen alias of Z (:43-44): Z receives gradients from the spatial kernel only.  Temporal
    hyperparameters: lengthscale_rbf, lengthscale_per, period = softplus(raw), outputscale = 7 + softplus(raw)."""

    def __init__(self, Z, log_ell_z, prior_c, prior_os, prior_lam, hyp_t=(1.0, 1.0, 1.0, 7.7), outputscale_s=0.644,
                 noise=0.011, outputscale_t_lower=7.0, learn_inducing_locations=True, include_prior=True):
        super().__init__()
        assert Z.shape[0] % 2 == 0, "M must be even (16-byte aligned column blocks of the n x 2M feature rows)"
        dev = Z.device
        self.os_t_lower = float(outputscale_t_lower)
        self.Z = torch.nn.Parameter(Z.clone(), requires_grad=learn_inducing_locations)
        self.log_ell_z = torch.nn.Parameter(log_ell_z.clone())
        lr, lp, per, os_t = (float(v) for v in hyp_t)
        self.raw_hyp_t = torch.nn.Parameter(torch.tensor(
            [_inv_softplus(lr), _inv_softplus(lp), _inv_softplus(per), _inv_softplus(os_t - self.os_t_lower)],
            dtype=torch.float64, device=dev))
        self.raw_outputscale = torch.nn.Parameter(torch.tensor([_inv_softplus(outputscale_s)], dtype=torch.float64,
                                                               device=dev))
        self.raw_noise = torch.nn.Parameter(torch.tensor([_inv_softplus(noise - 1e-4)], dtype=torch.float64, device=dev))
        self.register_buffer("prior_c", prior_c.clone())
        self.register_buffer("prior_os", prior_os.clone())
        self.register_buffer("prior_lam", prior_lam.clone())
        self.include_prior = include_prior

    def hyp_t(self):
        sp = _softplus(self.raw_hyp_t)
        return torch.cat([sp[:3], self.os_t_lower + sp[3:]])

    @staticmethod
    def _chol_ladder(Kzz, what):
        eye = torch.eye(Kzz.shape[0], dtype=torch.float64, device=Kzz.device)
        for jit in (0.0, 1e-8, 1e-7, 1e-6):  # psd_safe_cholesky ladder, keeping the jittered matrix (reused in Sigma)
            Kj = Kzz if jit == 0.0 else Kzz + jit * eye
            L, P, info = F.chol_inv(Kj)
            if int(info) == 0:
                return Kj, L, P
        raise RuntimeError("%s not positive definite after adding jitter up to 1e-6" % what)

    def _z_side(self):
        M = self.Z.shape[0]
        zs = self.Z[:, 1:3]
        zt = self.Z.detach()[:, 0].contiguous()  # frozen alias (spatio_temporal_models.py:43-44)
        D = 2
        ell_z = torch.exp(self.log_ell_z)
        eye = torch.eye(M, dtype=torch.float64, device=self.Z.device)
        alphas, lp = [], self.Z.new_zeros(())
        z_prior = self.Z[:, 0:2]  # the reference's prior term sees (time, lon): its closure passes the full (M,3) inducing
        # points and the prior's active_dims=(0,1) pick columns 0,1 (spatio_temporal_models.py:52-55, spatio_temporal_exp.py:111)
        for b in range(D):
            Kp = F.rbf_ard(zs, zs, self.prior_lam[b], self.prior_os[b]) + 1e-4 * eye
            Lb, Pb = F.psd_safe_chol_inv(Kp)
            r = self.log_ell_z[b] - self.prior_c[b]
            alphas.append(F.spd_solve(Pb, r))
            if self.include_prior:
                Kq = F.rbf_ard(z_prior, z_prior, self.prior_lam[b], self.prior_os[b]) + 1e-4 * eye
                Lq, Pq = F.psd_safe_chol_inv(Kq)
                lp = lp + (-0.5 * (r * F.spd_solve(Pq, r)).sum() - torch.log(torch.diagonal(Lq)).sum()
                           - 0.5 * M * LOG2PI) / M
        hyp = self.hyp_t()
        spatial = self._chol_ladder(F.gibbs_diag(zs, ell_z, zs, ell_z), "spatial Kzz")
        temporal = self._chol_ladder(ops.rbf_periodic(zt, zt, hyp), "temporal Kzz")
        return ell_z, torch.stack(alphas), hyp, zt, spatial, temporal, lp

    def _chunk_features(self, xc, zs, zt, hypd, ell_z, alpha, Fbuf):
        """Fbuf[:, :M] = K_t (outputscale included), Fbuf[:, M:] = unscaled Gibbs K_s; returns ell(x) of the chunk."""
        M = zs.shape[0]
        xt, xs = xc[:, 0].contiguous(), xc[:, 1:3].contiguous()
        ops.rbfper_fwd(xt, zt, hypd, out=Fbuf[:, :M])
        ell_x = ops.rbf_matvec_fwd(xs, zs, self.prior_lam, self.prior_os, alpha.unsqueeze(-1), bias=self.prior_c,
                                   apply_exp=True).squeeze(-1)
        ops.gibbs_diag_fwd(xs, ell_x, zs, ell_z, out=Fbuf[:, M:])
        return xt, xs, ell_x

    def _whiten(self, Fc, Gc, Pt, Ps):
        """Root rows of the chunk: G = [F_t P_t^T, F_s P_s^T] (the reference's k_ux1.matmul(inv_root),
        gibbs_kernels.py:225), two triangular DMMA GEMMs."""
        M = Pt.shape[0]
        ops.dgemm(Fc[:, :M], Pt, transB=True, tri_b=2, C=Gc[:, :M])
        ops.dgemm(Fc[:, M:], Ps, transB=True, tri_b=2, C=Gc[:, M:])

    def _pass1(self, x, y, chunk, zs, zt, hypd, ell_zd, alphad, Ptd, Psd, all_reduce):
        """Pass 1 over this rank's rows: W = G^T G, c = G^T y, y^T y of the whitened feature rows G = [F_t P_t^T, F_s P_s^T],
        summed over ranks by `all_reduce`.  Also returns the chunk buffers (F, G) for the caller's second pass."""
        dev = x.device
        n_loc = x.shape[0]
        M2 = 2 * self.Z.shape[0]
        W = torch.zeros(M2, M2, dtype=torch.float64, device=dev)
        c = torch.zeros(M2, dtype=torch.float64, device=dev)
        yy = torch.zeros((), dtype=torch.float64, device=dev)
        rows = min(chunk, n_loc)
        Fbuf = torch.empty(rows, M2, dtype=torch.float64, device=dev)
        Gbuf = torch.empty_like(Fbuf)
        Wc = torch.empty_like(W)
        for lo in range(0, n_loc, chunk):
            xc, yc = x[lo:lo + chunk], y[lo:lo + chunk].contiguous()
            Fc, Gc = Fbuf[:xc.shape[0]], Gbuf[:xc.shape[0]]
            self._chunk_features(xc, zs, zt, hypd, ell_zd, alphad, Fc)
            self._whiten(Fc, Gc, Ptd, Psd)
            W += _syrk(Gc, Wc, getattr(self, 'use_i8', True))
            ops.colwsum(Gc, w=yc, out=c)
            yy += (yc * yc).sum()
        if all_reduce is not None:
            packed = torch.cat([W.reshape(-1), c, yy.reshape(1)])
            all_reduce(packed)
            W, c, yy = packed[:M2 * M2].reshape(M2, M2), packed[M2 * M2:M2 * M2 + M2], packed[-1]
        return W, c, yy, Fbuf, Gbuf

    @torch.no_grad()
    def posterior(self, x, y, *, chunk: int = 32768, n_total: Optional[int] = None, all_reduce=None) -> "SGPRPosterior":
        """The collapsed posterior of the spatio-temporal model at the current parameters (the literal=False predictive of
        the reference, spatio_temporal_exp.py's default), from pass 1 of neg_objective_and_grad over this rank's rows,
        all-reduced the same way.  Returns a snapshot that later parameter updates do not change.  With D = diag(I_M,
        sqrt(s) I_M), B = I + D W D / noise, P_B = chol(B)^-1, P = blockdiag(P_t, P_s) and features k = [k_t | k_s]:
            mean = k^T u,  u = P^T D B^-1 D c / noise,
            var_f = max(os_t - |P_t k_t|^2, 0) + s max(1 - |P_s k_s|^2, 0) + |V k|^2,   V = P_B D P (lower triangular).
        `n_total` is accepted for symmetry with neg_objective_and_grad; the posterior does not depend on it."""
        del n_total
        M = self.Z.shape[0]
        M2 = 2 * M
        ell_z, alpha, hyp, zt, (_, _, Ps), (_, _, Pt), _ = self._z_side()
        ell_z, alpha, hyp = ell_z.contiguous(), alpha.contiguous(), hyp.contiguous()
        zs = self.Z[:, 1:3].contiguous()
        W, c, _, _, _ = self._pass1(x, y, chunk, zs, zt, hyp, ell_z, alpha, Pt, Ps, all_reduce)
        s = _softplus(self.raw_outputscale).reshape(())
        noise = (1e-4 + _softplus(self.raw_noise)).reshape(())
        sv = torch.cat([torch.ones(M, dtype=torch.float64, device=x.device), torch.sqrt(s).expand(M)])
        Bm = torch.eye(M2, dtype=torch.float64, device=x.device) + 0.5 * (W + W.T) * sv[:, None] * sv[None, :] / noise
        _, PB = F.psd_safe_chol_inv(Bm)
        w = F.matmul(PB.T, F.matmul(PB, c * sv)) * sv / noise          # D B^-1 D c / noise
        u = torch.cat([F.matmul(Pt.T, w[:M]), F.matmul(Ps.T, w[M:])])
        P = torch.zeros(M2, M2, dtype=torch.float64, device=x.device)  # blockdiag(P_t, P_s)
        P[:M, :M] = Pt
        P[M:, M:] = Ps
        V = ops.dgemm(PB, P * sv[:, None], tri_a=1, tri_b=1, out_tri=1, C=torch.zeros_like(P))
        return SGPRPosterior(self, "st", P=P, V=V, u=u, s=s, noise=noise, ell_z=ell_z, alpha=alpha, hyp=hyp, zt=zt,
                             use_i8=getattr(self, "use_i8", True))

    def neg_objective_and_grad(self, x, y, chunk: int = 32768, n_total: Optional[int] = None, all_reduce=None):
        """As SGPRGibbsStream.neg_objective_and_grad, for x (n, 3) = (time, lon, lat).

        Numerics: Kzz of the temporal kernel (M inducing times on a smooth 1-D kernel) is nearly singular, and at
        N ~ 4e6 rows the unwhitened Gram matrix F^T F / noise has norm ~1e12, so `Kzz + F^T F / noise` cannot be
        factored in fp64.  Rows are therefore whitened chunk by chunk BEFORE they are accumulated, G = F L^-T, exactly
        as the reference forms its root; then B = I + D G^T G D / noise has eigenvalues >= 1 and the log-determinants of
        Kzz cancel analytically.  Cost per row: 22 M^2 flop for both passes instead of 12 M^2."""
        dev = x.device
        n_loc = x.shape[0]
        n = n_total if n_total is not None else n_loc
        M = self.Z.shape[0]
        M2 = 2 * M
        ell_z, alpha, hyp, zt, (_, _, Ps), (_, _, Pt), lp = self._z_side()
        ell_zd, alphad, hypd = ell_z.detach().contiguous(), alpha.detach().contiguous(), hyp.detach().contiguous()
        Ptd, Psd = Pt.detach(), Ps.detach()
        zs = self.Z.detach()[:, 1:3].contiguous()

        W, c, yy, Fbuf, Gbuf = self._pass1(x, y, chunk, zs, zt, hypd, ell_zd, alphad, Ptd, Psd, all_reduce)
        W = W.clone().requires_grad_(True)
        c = c.clone().requires_grad_(True)

        # ---- 2M x 2M algebra: B = I + D W D / noise, D = diag(1, sqrt(s))
        s = _softplus(self.raw_outputscale).reshape(())
        noise = (1e-4 + _softplus(self.raw_noise)).reshape(())
        sv = torch.cat([torch.ones(M, dtype=torch.float64, device=dev), torch.sqrt(s).expand(M)])
        Ws = 0.5 * (W + W.T) * sv[:, None] * sv[None, :]
        cs = c * sv
        Bm = torch.eye(M2, dtype=torch.float64, device=dev) + Ws / noise
        LB, PB = F.psd_safe_chol_inv(Bm)
        w = F.matmul(PB, cs)
        quad = yy / noise - (w * w).sum() / (noise * noise)
        logdet = 2.0 * torch.log(torch.diagonal(LB)).sum() + n * torch.log(noise)
        ll = -0.5 * (quad + logdet + n * LOG2PI)
        dW_ = torch.diagonal(W)
        trace_t = -0.5 * (n * hyp[3] - dW_[:M].sum()) / noise
        trace_s = -0.5 * (n - dW_[M:].sum()) / noise  # unscaled: GibbsSafeScaleKernel wraps the Nystrom kernel
        obj = (ll + trace_t + trace_s + lp) / n
        loss = -obj
        dW, dc = torch.autograd.grad(loss, [W, c], retain_graph=True)
        dW2 = (dW + dW.T).contiguous()
        dc = dc.contiguous()

        # ---- pass 2: dG = G (dW + dW^T) + y dc^T;  dF = dG P (to the analytic kernel backwards);  dP += dG^T F
        d_ell_z = torch.zeros_like(ell_zd)
        dZs = torch.zeros(M, 2, dtype=torch.float64, device=dev)
        dalpha = torch.zeros(2, M, 1, dtype=torch.float64, device=dev)
        dhyp = torch.zeros(4, dtype=torch.float64, device=dev)
        dPt = torch.zeros(M, M, dtype=torch.float64, device=dev)
        dPs = torch.zeros(M, M, dtype=torch.float64, device=dev)
        Tbuf = torch.empty_like(Fbuf)
        need_dz = self.Z.requires_grad
        for lo in range(0, n_loc, chunk):
            xc, yc = x[lo:lo + chunk], y[lo:lo + chunk].contiguous()
            Fc, Gc, Tc = Fbuf[:xc.shape[0]], Gbuf[:xc.shape[0]], Tbuf[:xc.shape[0]]
            xt, xs, ell_x = self._chunk_features(xc, zs, zt, hypd, ell_zd, alphad, Fc)
            self._whiten(Fc, Gc, Ptd, Psd)
            _rowmul(Gc, dW2, Tc, getattr(self, 'use_i8', True))
            Tc.addcmul_(yc.unsqueeze(1), dc.unsqueeze(0))
            ops.dgemm(Tc[:, :M], Fc[:, :M], transA=True, beta=1.0, C=dPt)
            ops.dgemm(Tc[:, M:], Fc[:, M:], transA=True, beta=1.0, C=dPs)
            dFc = Gc  # G is no longer needed: reuse its storage for dF
            ops.dgemm(Tc[:, :M], Ptd, tri_b=1, C=dFc[:, :M])
            ops.dgemm(Tc[:, M:], Psd, tri_b=1, C=dFc[:, M:])
            g4, _ = ops.rbfper_bwd(xt, zt, hypd, dFc[:, :M])
            dhyp += g4
            r = ops.gibbs_diag_bwd(xs, ell_x, zs, ell_zd, None, G=dFc[:, M:], need_dx2=need_dz)
            d_ell_z += r["d_ell2"]
            dlog = (r["d_ell1"] * ell_x).unsqueeze(-1)
            da, dzf = ops.rbf_matvec_bwd(xs, zs, self.prior_lam, self.prior_os, alphad.unsqueeze(-1), dlog, need_dz=need_dz)
            dalpha += da
            if need_dz:
                dZs += r["d_x2"] + dzf
        if all_reduce is not None:
            parts = [d_ell_z, dZs, dalpha, dhyp, dPt, dPs]
            packed = torch.cat([t.reshape(-1) for t in parts])
            all_reduce(packed)
            out, off = [], 0
            for t in parts:
                out.append(packed[off:off + t.numel()].reshape(t.shape))
                off += t.numel()
            d_ell_z, dZs, dalpha, dhyp, dPt, dPs = out

        for p_ in self.parameters():
            p_.grad = None
        torch.autograd.backward([loss, alpha, hyp, Pt, Ps],
                                [torch.ones_like(loss), dalpha.squeeze(-1), dhyp, torch.tril(dPt), torch.tril(dPs)])
        with torch.no_grad():
            self.log_ell_z.grad += d_ell_z * ell_zd
            if need_dz:
                self.Z.grad[:, 1:3] += dZs
        return loss.detach()


class SGPRPosterior:
    """Snapshot of a streamed SGPR posterior, returned by SGPRGibbsStream.posterior ("diag") and
    SGPRSpatioTemporalStream.posterior ("st").  It holds copies of everything the predictive and the sampler need (Z, the
    lengthscale field's interpolation weights, u, P -- as digit planes when the feature width W is a multiple of 128 -- and V
    in FP64, plus its planes on that path), so later optimiser steps on the model do not change its predictions or draws.
    V costs 8 W^2 bytes in FP64 (134 MB at W = 4096); sample() needs it to form W^T = E^T V."""

    def __init__(self, model, kind, *, P, V, u, s, noise, ell_z, alpha, use_i8, hyp=None, zt=None):
        self.kind = kind
        self.M = model.Z.shape[0]
        self.width = P.shape[0]  # M (diag) or 2M (st): the feature columns of a test row
        self.Z = model.Z.detach().clone()
        self.zs = self.Z[:, 1:3].contiguous() if kind == "st" else self.Z
        self.prior_c, self.prior_os, self.prior_lam = (b.detach().clone() for b in
                                                       (model.prior_c, model.prior_os, model.prior_lam))
        self.ell_z, self.alpha, self.u = ell_z.detach().clone(), alpha.detach().clone(), u.detach().contiguous().clone()
        self.s, self.noise = s.detach().clone(), noise.detach().clone()
        self.hyp = hyp.detach().clone() if hyp is not None else None
        self.zt = zt.detach().clone() if zt is not None else None
        self.digits = bool(use_i8) and self.width % 128 == 0
        self.V = V.detach().clone()
        if self.digits:
            self.planes = []
            for Mx in (P, V):  # B operands of npgp_o8_trinorm_digits: block_rows 64, per-row exponents
                d = torch.empty(ops.digits_bytes(self.width, self.width, 64), dtype=torch.uint8, device=P.device)
                e = torch.empty(self.width, dtype=torch.int32, device=P.device)
                ops.o8_slice_rows(Mx.contiguous(), 64, d, e)
                self.planes.append((d, e))
            self.one = torch.ones((), dtype=torch.float64, device=P.device)  # bound of the unscaled Gibbs entries
        else:
            M = self.M
            self.Pblocks = [P[:M, :M].contiguous(), P[M:, M:].contiguous()] if kind == "st" else [P.detach().clone()]

    def _row_buffers(self, xs, chunk):
        """Buffers of the row pass (_row_chunk) over xs in chunks of up to `chunk` rows, allocated once per call."""
        n, dev = xs.shape[0], xs.device
        f64 = dict(dtype=torch.float64, device=dev)
        st = self.kind == "st"
        M, W = self.M, self.width
        rows = min(chunk, n)
        cdiv = lambda a, b: (a + b - 1) // b  # noqa: E731
        b = dict(D=2 if st else self.Z.shape[1], rows=rows)
        b["nb_t"] = (M // 64 if self.digits else cdiv(M, 64)) if st else 0
        nbn = W // 64 if self.digits else (2 if st else 1) * cdiv(M, 64)
        b["qn"] = torch.empty(nbn, rows, **f64)
        b["ell"] = torch.empty(b["D"] * rows, **f64)
        if st:
            b["xt"], b["xs"] = xs[:, 0].contiguous(), xs[:, 1:3].contiguous()
            b["F"] = torch.empty(rows, W, **f64)
        else:
            b["xs"] = xs
        if self.digits:
            b["Ad"] = torch.empty(ops.digits_bytes(rows, W, 128), dtype=torch.uint8, device=dev)
            if st:
                b["Ae"] = torch.empty(cdiv(rows, 128) * 128, dtype=torch.int32, device=dev)
            else:
                sizes = {rows, n - (n - 1) // chunk * chunk}
                b["ku"] = torch.empty(max(ops.gibbs_digits_splits(r, M) for r in sizes) * rows, **f64)
        else:
            b["G"] = torch.empty(rows, W, **f64)
            if not st:
                b["K"] = torch.empty(rows, M, **f64)
        return b

    def _row_chunk(self, b, lo, nc, mean):
        """The part of a chunk of rows lo .. lo + nc that predictive() and sample() share: the lengthscale field, the feature
        rows k(x) (FP64 and/or digit planes in b), the mean k^T u into `mean` and the partials of |P k|^2 into b["qn"].
        Returns (ell(x) (D, nc), the FP64 feature rows (nc, W) or None on the diagonal model's digit path)."""
        st = self.kind == "st"
        M, W, D, qn = self.M, self.width, b["D"], b["qn"]
        ell = b["ell"][:D * nc].view(D, nc, 1)
        xc = b["xs"][lo:lo + nc]
        ops.rbf_matvec_fwd(xc, self.zs, self.prior_lam, self.prior_os, self.alpha.unsqueeze(-1), bias=self.prior_c,
                           apply_exp=True, out=ell)
        ell_x = ell.view(D, nc)
        if st:
            Fc = b["F"][:nc]
            ops.rbfper_fwd(b["xt"][lo:lo + nc], self.zt, self.hyp, out=Fc[:, :M])
            ops.gibbs_diag_fwd(xc, ell_x, self.zs, self.ell_z, out=Fc[:, M:])
            ops.gemv_n(Fc, self.u, out=mean)
            if self.digits:
                ops.o8_slice_rows(Fc, 128, b["Ad"], b["Ae"])
                ops.o8_trinorm_digits(nc, W, W, b["Ad"], None, *self.planes[0], qn, Ms=M, a_expo=b["Ae"])
            else:
                Gc, nb_t = b["G"][:nc], b["nb_t"]
                for h, Ph in enumerate(self.Pblocks):
                    cols = slice(h * M, (h + 1) * M)
                    ops.dgemm(Fc[:, cols], Ph, transB=True, tri_b=2, C=Gc[:, cols])
                    ops.sgpr_rownorm_parts(Gc[:, cols], qn[h * nb_t:(h + 1) * nb_t])
            return ell_x, Fc
        if self.digits:
            kup = b["ku"][:ops.gibbs_digits_splits(nc, M) * nc].view(-1, nc)
            ops.gibbs_diag_fwd_digits(xc, ell_x, self.Z, self.ell_z, self.one, b["Ad"], u=self.u, Ku_part=kup)
            ops.o8_sum_partials(kup, out=mean)
            ops.o8_trinorm_digits(nc, M, M, b["Ad"], self.one, *self.planes[0], qn)
            return ell_x, None
        K = ops.gibbs_diag_fwd(xc, ell_x, self.Z, self.ell_z, out=b["K"][:nc])
        ops.gemv_n(K, self.u, out=mean)
        ops.sgpr_rownorm_parts(ops.dgemm(K, self.Pblocks[0], transB=True, tri_b=2, C=b["G"][:nc]), qn)
        return ell_x, K

    @torch.no_grad()
    def predictive(self, xs, y=None, *, field: bool = False, chunk: int = 65536):
        """Posterior marginals at the rows xs (n, D), streamed in chunks of `chunk` rows: svgp.Predictive with mean, var
        (of f), var_y = var + noise, field (field=True): ell(x) (D, n) on the Gibbs columns, and with y: lpd = log N(y |
        mean, var_y) and sums = [sum (y - mean)^2, sum -lpd, n].  Buffers are allocated once per call, the chunk loop does
        not synchronise with the host, and every reduction has a fixed order.  Rows may be sharded over ranks with no
        collective: one all-reduce of the three sums gives the global RMSE and NLPD."""
        from .svgp import Predictive
        xs = xs.contiguous()
        n = xs.shape[0]
        dev = xs.device
        f64 = dict(dtype=torch.float64, device=dev)
        st = self.kind == "st"
        W = self.width
        D = 2 if st else self.Z.shape[1]
        mean, var, var_y = (torch.empty(n, **f64) for _ in range(3))
        fld = torch.empty(D, n, **f64) if field else None
        lpd = sums = None
        if y is not None:
            y = y.contiguous()
            lpd, sums = torch.empty(n, **f64), torch.zeros(3, **f64)
        if n == 0:
            return Predictive(mean, var, var_y, fld, lpd, sums)
        b = self._row_buffers(xs, chunk)
        qn, nb_t = b["qn"], b["nb_t"]
        qv = torch.empty((W + 63) // 64, b["rows"], **f64)
        work = ops.sgpr_predict_workspace(b["rows"], dev) if y is not None else None
        for lo in range(0, n, chunk):
            nc = min(chunk, n - lo)
            mc = mean[lo:lo + nc]
            ell_x, feats = self._row_chunk(b, lo, nc, mc)
            if self.digits:
                ops.o8_trinorm_digits(nc, W, W, b["Ad"], None if st else self.one, *self.planes[1], qv,
                                      a_expo=b["Ae"] if st else None)
            else:
                ops.sgpr_rownorm_parts(ops.dgemm(feats, self.V, transB=True, tri_b=2, C=b["G"][:nc]), qv)
            if field:
                fld[:, lo:lo + nc] = ell_x
            ops.sgpr_predict_finish(qn, nb_t, qv, self.s, self.noise, var[lo:lo + nc], os_t=self.hyp[3:] if st else None,
                                    mean=mc, y=y[lo:lo + nc] if y is not None else None, var_y=var_y[lo:lo + nc],
                                    lpd=lpd[lo:lo + nc] if y is not None else None, sums=sums, work=work)
        return Predictive(mean, var, var_y, fld, lpd, sums)

    @torch.no_grad()
    def sample(self, xs, num_samples: int, *, seed: int = 0, noise: bool = False, row_offset: int = 0,
               chunk: int = 65536) -> torch.Tensor:
        """num_samples posterior draws of f (noise=True: of y) at the rows xs (n, D), correlated across rows: (num_samples,
        n), streamed in chunks of `chunk` rows.  The draws are exact samples of the joint predictive of posterior(), i.e. of
        the reference's eval-mode predictive with the low-rank root (for the spatio-temporal model its literal=False form,
        not the default literal=True one, whose dense-row factors give a covariance of another form):
            f_s(x) = k(x)^T u + (V k(x))^T e_s + sqrt(r(x)) xi_s(x),   e_s ~ N(0, I_W),  xi_s(x) ~ N(0, 1)
            Cov(f(x), f(x')) = (V k(x))^T (V k(x')) + delta(x, x') r(x),   r(x) = predictive().var - |V k(x)|^2
        with r(x) = [st] max(os_t - |P_t k_t|^2, 0) + s max(1 - |P_s k_s|^2, 0).  noise=True adds the noise variance to r.
        The mean term is predictive().mean.  Keys as SVGPGibbs.sample: e_s[j] = normal(seed, (s << 32) + j) and xi_s(row) =
        normal(seed, 2^63 + (s << 48) + row_offset + i), so draw s does not depend on num_samples and rows sharded over ranks
        with their global row_offset are parts of one joint draw (up to the rounding of the M x M algebra that posterior()
        replicates after its all-reduce).  Per call: E^T (64 ceil(S / 64) x W), W^T = E^T V and its digit planes, then per
        chunk the rows as in predictive() without its V pass, K W^T^T and one finishing kernel; buffers are allocated once
        per call and the chunk loop does not synchronise with the host.  For the same snapshot, rows, chunking and seed the
        draws are bitwise reproducible below W = 512; from there on npgp_dgemm may split the product E^T V over its inner
        dimension with FP64 atomics (small outputs with a long inner dimension), and two calls then agree to rounding."""
        S = int(num_samples)
        if not 1 <= S <= 1024:
            raise ValueError("num_samples must be in 1 .. 1024 (got %d)" % S)
        xs = xs.contiguous()
        n = xs.shape[0]
        if row_offset < 0 or row_offset + n > 1 << 48:
            raise ValueError("rows row_offset .. row_offset + n must lie in [0, 2^48) (got %d + %d)" % (row_offset, n))
        dev = xs.device
        f64 = dict(dtype=torch.float64, device=dev)
        out = torch.empty(S, n, **f64)
        if n == 0:
            return out
        st = self.kind == "st"
        W, Sp = self.width, (S + 63) // 64 * 64
        Wt = ops.dgemm(ops.sample_normals(W, S, seed, torch.empty(Sp, W, **f64)), self.V, tri_b=1)  # W^T = E^T V
        b = self._row_buffers(xs, chunk)
        if self.digits:
            Wd = torch.empty(ops.digits_bytes(Sp, W, 64), dtype=torch.uint8, device=dev)
            We = torch.empty(Sp, dtype=torch.int32, device=dev)
            ops.o8_slice_rows(Wt, 64, Wd, We)
        mean = torch.empty(b["rows"], **f64)
        Fbuf = torch.empty(b["rows"], Sp, **f64)
        for lo in range(0, n, chunk):
            nc = min(chunk, n - lo)
            mc, Fc = mean[:nc], Fbuf[:nc]
            _, feats = self._row_chunk(b, lo, nc, mc)
            if self.digits:
                ops.o8_gemm_digits(nc, Sp, W, b["Ad"], None if st else self.one, Wd, We, Fc, a_expo=b["Ae"] if st else None)
            else:
                ops.dgemm(feats, Wt, transB=True, C=Fc)
            ops.sgpr_sample_finish(mc, b["qn"], b["nb_t"], Fc, S, self.s, self.noise, out[:, lo:lo + nc],
                                   os_t=self.hyp[3:] if st else None, add_noise=noise, seed=seed, row0=row_offset + lo)
        return out
