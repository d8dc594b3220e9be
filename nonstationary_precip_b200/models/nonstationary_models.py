"""Mirror of the reference's models/nonstationary_models.py (GP models using Gibbs kernels) on the npgp kernels.

  DiagonalExactGP(train_x, train_y, likelihood, prior, num_dim=1)      reference models/nonstationary_models.py:22-62
  DiagonalSparseGP(train_x, train_y, likelihood, prior, z, num_dim=1)  reference models/nonstationary_models.py:64-153

`forward(x)` returns the prior MultivariateNormal at the training inputs (to be scored by ExactMarginalLogLikelihood),
`predict(x_new)` the predictive distribution, exactly as in the reference, and `posterior()` a snapshot that predicts and
draws correlated sample fields at any number of rows (sgpr.SGPRPosterior)."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from .. import functional as F
from .. import ops
from ..gp_base import ExactGP, LowRankRootCovar, MultivariateNormal, ZeroMean
from ..sgpr import SGPRGibbsStream, SGPRPosterior
from .gibbs_kernels import GibbsKernel, GibbsSafeScaleKernel, InducingGibbsKernel


class DiagonalExactGP(ExactGP):
    """MAP inference of a diagonal-Gibbs GP over the per-training-point log-lengthscales `log_ell_train_x` (D, n)."""

    def __init__(self, train_x, train_y, likelihood, prior, num_dim=1):
        super().__init__(train_x, train_y, likelihood)
        self.mean_module = ZeroMean()
        self.covar_module = GibbsSafeScaleKernel(GibbsKernel(lengthscale_prior=prior, ard_num_dims=num_dim))
        prior_mean = self.covar_module.base_kernel.lengthscale_prior.mean_module(self.train_inputs[0])
        self.register_parameter("log_ell_train_x", torch.nn.Parameter(prior_mean.detach().clone()))
        self.register_prior("ell_train_prior", self.covar_module.base_kernel.lengthscale_prior,
                            lambda module: (module.train_inputs[0], module.log_ell_train_x))

    def forward(self, x):
        mean = self.mean_module(x)
        covar = self.covar_module(x, ell1=torch.exp(self.log_ell_train_x))
        return MultivariateNormal(mean, covar)

    def predict(self, x_new):
        """Predictive at x_new given the lengthscales at the training points (reference :45-62): full covariance
        K_ss - K_sx (K_xx + noise I)^-1 K_xs + 1e-4 I."""
        x = self.train_inputs[0]
        ell = torch.exp(self.log_ell_train_x)
        noise = self.likelihood.noise.reshape(())
        K_xx = self.covar_module(x, ell1=ell)
        ell2 = self.covar_module.base_kernel.lengthscale_prior.conditional_sample(x_new, given=(x, ell))
        K_ss = self.covar_module(x_new, ell1=ell2)
        K_sx = self.covar_module(x_new, x, ell1=ell2, ell2=ell)
        n = K_xx.shape[-1]
        _, P = F.psd_safe_chol_inv(K_xx + noise * torch.eye(n, dtype=x.dtype, device=x.device))
        A = F.matmul(K_sx, P.T)  # K_sx L^-T
        mu = F.matmul(A, F.matmul(P, self.train_targets))
        sigma = K_ss - F.matmul(A, A.T)
        ns = K_ss.shape[-1]
        return MultivariateNormal(mu, sigma + 1e-4 * torch.eye(ns, dtype=x.dtype, device=x.device))

    @torch.no_grad()
    def posterior(self, *, knots=None) -> SGPRPosterior:
        """Snapshot of the posterior at the current parameters for prediction and sample fields at any number of rows
        (sgpr.SGPRPosterior: .predictive(xs, y=None, *, field, chunk), .sample(xs, num_samples, *, seed, noise, row_offset,
        chunk)); predict() builds n* x n* matrices.  With the unscaled kernel k, outputscale s, noise sigma^2,
        tau = sigma^2 / s and P_y = chol(K_XX + tau I)^-1 the marginals are those of predict():
            mean = k^T u,  u = P_y^T P_y y,    var_f = s max(1 - |P_y k|^2, 0) + 1e-4,    var_y = var_f + sigma^2,
        where k^T (K + tau I)^-1 k < 1, so the clamp changes nothing beyond rounding; the field at new rows is the prior's
        conditional mean given the training lengthscales, as in predict().
        The draws are a predictive process on the knots U = [X; knots] (knots (m, D), optional; their lengthscales come from
        the same field): the collapsed SGPR posterior with inducing set U, which contains the training rows.  With
        P_U = chol(K_UU + j I)^-1 (j the first of 0, 1e-8, 1e-7, 1e-6 that factors), W = P_U K_UX K_XU P_U^T,
        B = I + (s / sigma^2) W and V = sqrt(s) chol(B)^-1 P_U,
            f_s(x) = mean(x) + (V k_U(x))^T e_s + sqrt(s max(1 - |P_U k_U(x)|^2, 0) + 1e-4 [+ sigma^2 if noise]) xi_s(x).
        With j = 0 each marginal equals var_f; the covariance departs from predict()'s only by the off-diagonal Nystrom
        residual s (k(x, x') - k_U(x)^T K_UU^-1 k_U(x')), set to zero, which knots make smaller.  The columns are padded to
        a multiple of 128 (copies of a training row, zero rows and columns in P_y, P_U, V and zeros in u) so that any n takes
        the int8 digit path (use_i8 = False: the FP64 path); the results do not depend on the padding beyond rounding."""
        x = self.train_inputs[0]
        n, D = x.shape
        prior = self.covar_module.base_kernel.lengthscale_prior
        if knots is not None and (knots.dim() != 2 or knots.shape[1] != D):
            raise ValueError("knots must have shape (m, %d) (got %s)" % (D, tuple(knots.shape)))
        m = 0 if knots is None else knots.shape[0]
        Wp = -(-(n + m) // 128) * 128
        if Wp > 16384:
            raise ValueError("n + m = %d padded to %d exceeds the digit engine's 16384 columns" % (n + m, Wp))
        f64 = dict(dtype=torch.float64, device=x.device)
        ell = torch.exp(self.log_ell_train_x)
        s = self.covar_module.outputscale.reshape(()).clone()
        noise = self.likelihood.noise.reshape(()).clone()
        tau = noise / s
        U, ell_u = x, ell
        if m:
            knots = knots.to(**f64).contiguous()
            U = torch.cat([x, knots])
            ell_u = torch.cat([ell, prior.conditional_sample(knots, given=(x, ell))], 1)
        K = F.gibbs_diag(U, ell_u, U, ell_u)
        eye = torch.eye(n + m, **f64)
        _, Py = F.psd_safe_chol_inv(K[:n, :n] + tau * eye[:n, :n])
        u = F.spd_solve(Py, self.train_targets)
        tau_h = float(tau)
        for jit in (0.0, 1e-8, 1e-7, 1e-6):  # psd_safe_cholesky ladder, as SGPRGibbsStream._z_side
            if jit >= tau_h:
                raise ValueError("K_UU needs jitter %g, not below tau = noise / outputscale = %g" % (jit, tau_h))
            _, PU, info = F.chol_inv(K + jit * eye if jit else K)
            if int(info) == 0:
                break
        else:
            raise ValueError("K_UU not positive definite after adding jitter up to 1e-6")
        G = F.matmul(K[:n], PU.T)  # K_XU P_U^T
        Bm = eye + (s / noise) * F.matmul(G.T, G)
        _, PB = F.psd_safe_chol_inv(0.5 * (Bm + Bm.T))
        V = ops.dgemm(F._aligned(PB), F._aligned(PU), tri_a=1, tri_b=1, out_tri=1, C=torch.zeros_like(PU))
        V *= torch.sqrt(s)

        def pad(A, rows, cols):
            out = torch.zeros(rows, cols, **f64)
            out[:A.shape[0], :A.shape[1]] = A
            return out
        up = torch.zeros(Wp, **f64)
        up[:n] = u
        c, os_, lam = prior._hypers()
        cols = SimpleNamespace(Z=torch.cat([U, x[:1].expand(Wp - n - m, D)]), prior_c=c, prior_os=os_, prior_lam=lam)
        return SGPRPosterior(cols, "exact", P=pad(Py, Wp, Wp), V=pad(V, Wp, Wp), u=up, s=s, noise=noise,
                             ell_z=torch.cat([ell_u, ell[:, :1].expand(D, Wp - n - m)], 1).contiguous(),
                             alpha=prior.conditional_weights(x, ell), use_i8=getattr(self, "use_i8", True), field_x=x,
                             P_draws=pad(PU, Wp, Wp), add_var=1e-4)


class DiagonalSparseGP(ExactGP):
    """MAP inference of the sparse (SGPR) Gibbs GP over the log-lengthscales at the inducing points `log_ell_z` (D, M)."""

    def __init__(self, train_x, train_y, likelihood, prior, z, num_dim=1):
        super().__init__(train_x, train_y, likelihood)
        self.mean_module = ZeroMean()
        self.covar_module = GibbsSafeScaleKernel(
            InducingGibbsKernel(GibbsKernel(lengthscale_prior=prior, ard_num_dims=num_dim), z, likelihood))
        zz = z.unsqueeze(-1) if z.dim() == 1 else z
        prior_mean = self.covar_module.base_kernel.base_kernel.lengthscale_prior.mean_module(zz)
        self.register_parameter("log_ell_z", torch.nn.Parameter(prior_mean.detach().clone()))
        self.register_prior("ell_z_prior", self.covar_module.base_kernel.base_kernel.lengthscale_prior,
                            lambda module: (module.covar_module.base_kernel.inducing_points, module.log_ell_z))

    def forward(self, x, ell=None):
        mean = self.mean_module(x)
        covar = self.covar_module(x, ell=torch.exp(self.log_ell_z))
        return MultivariateNormal(mean, covar)

    def predict(self, x_new):
        """Predictive at x_new (reference :91-153): joint low-rank root over [train; test], B = I + A A^T,
        mean = L B^-1 A y / sigma, covariance = K_** - L (I - B^-1) L^T.  As the reference warns, only the marginals
        are meaningful."""
        x = self.train_inputs[0]
        if x_new.dim() == 1:
            x_new = x_new.unsqueeze(-1)
        n = x.shape[-2]
        full_output = self.forward(torch.cat([x, x_new], dim=-2))
        full_covar = full_output.lazy_covariance_matrix
        assert isinstance(full_covar, LowRankRootCovar)
        root = full_covar.root
        noise = self.likelihood.noise.reshape(())
        L = root[n:]
        At = root[:n] / torch.sqrt(noise)
        M = root.shape[-1]
        eye = torch.eye(M, dtype=x.dtype, device=x.device)
        B = eye + F.matmul(At.T, At)
        LB, PB = F.psd_safe_chol_inv(B)
        Binv = F.matmul(PB.T, PB)
        mean = F.matmul(L, F.matmul(Binv, F.matmul(At.T, self.train_targets))) / torch.sqrt(noise) \
            + full_output.loc[n:]
        test_test = F.matmul(L, L.T)
        if full_covar.added_diag is not None:
            test_test = test_test + torch.diag(full_covar.added_diag[n:])
        covar = test_test - F.matmul(L, F.matmul(eye - Binv, L.T))
        return MultivariateNormal(mean, covar)

    @torch.no_grad()
    def posterior(self) -> SGPRPosterior:
        """Snapshot of the posterior at the current parameters for prediction and sample fields at any number of rows: the
        one SGPRGibbsStream.posterior returns for this model's inducing points, lengthscales, outputscale, noise, prior and
        training data.  Its marginals are those of predict() and its draws are exact samples of predict()'s joint
        Lr B^-1 Lr^T + diag(clamp(s - |Lr|^2, 0)).  Inducing sets whose size is not a multiple of 128 take the FP64 path."""
        x, y = self.train_inputs[0], self.train_targets
        ind = self.covar_module.base_kernel
        prior = ind.base_kernel.lengthscale_prior
        c, os_, lam = prior._hypers()
        stream = SGPRGibbsStream(ind.inducing_points.detach(), self.log_ell_z.detach(), c, os_, lam,
                                 outputscale=float(self.covar_module.outputscale), noise=float(self.likelihood.noise),
                                 learn_inducing_locations=False, include_prior=False)
        stream.use_i8 = getattr(self, "use_i8", True)
        return stream.posterior(x.contiguous(), y.contiguous())
