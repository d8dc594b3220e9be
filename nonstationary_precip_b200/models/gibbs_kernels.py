"""Mirror of the reference's models/gibbs_kernels.py on the npgp CUDA kernels: same class names, constructor and call
signatures, parameter names and error behaviour; the arithmetic runs in fused kernels with analytic backward.

  PositivePriorProcess, LogNormalPriorProcess   reference models/gibbs_kernels.py:35-109
  GibbsKernel                                   reference models/gibbs_kernels.py:111-162
  GibbsSafeScaleKernel                          reference models/gibbs_kernels.py:164-168
  InducingGibbsKernel, InducingGibbsKernelST    reference models/gibbs_kernels.py:171-363
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

from .. import functional as F
from ..gp_base import (ConstantMean, InducingPointKernelAddedLossTerm, Kernel, LowRankRootCovar, Module,
                       MultivariateNormal, RBFKernel, ScaleKernel)


class PositivePriorProcess(Module):
    """Base class for lengthscale prior processes (reference :35-59)."""

    def forward(self, x):
        raise NotImplementedError

    def sample(self, x, **kwargs):
        raise NotImplementedError

    def conditional_sample(self, x, given, **kwargs):
        raise NotImplementedError


class LogNormalPriorProcess(PositivePriorProcess):
    """D independent GPs on the log-lengthscale (reference :61-109): ConstantMean and scaled ARD-RBF, both with batch
    shape (D,).  `conditional_sample` returns exp of the conditional mean, evaluated matrix free."""

    def __init__(self, input_dim: int = 1, covariance_function=None, active_dims=None):
        super().__init__()
        self.input_dim = input_dim
        self.mean_module = ConstantMean(batch_shape=torch.Size((input_dim,)))
        if covariance_function is None:
            covariance_function = ScaleKernel(
                RBFKernel(ard_num_dims=input_dim, batch_shape=torch.Size((input_dim,)), active_dims=active_dims),
                batch_shape=torch.Size((input_dim,)), active_dims=active_dims)
        self.covar_module = covariance_function

    def _active(self, x):
        """gpytorch.Kernel.__call__ semantics of `self.covar_module(x)`: the (outer) kernel's active_dims select the
        input columns once; with active_dims=(0,1) a 2-column input passes unchanged and a 3-column one keeps 0,1."""
        ad = getattr(self.covar_module, "active_dims", None)
        if ad is None:
            return x
        return x.index_select(-1, ad.to(x.device)).contiguous()

    def _hypers(self):
        D = self.input_dim
        lam = self.covar_module.base_kernel.lengthscale.reshape(D, -1)
        if lam.shape[1] == 1:
            lam = lam.expand(D, D)
        return self.mean_module.constant.reshape(D), self.covar_module.outputscale.reshape(D), lam.contiguous()

    def _prior_cov(self, x):
        c, os, lam = self._hypers()
        x = self._active(x)
        return torch.stack([F.rbf_ard(x, x, lam[b], os[b]) for b in range(self.input_dim)])

    def forward(self, x):
        """Distribution of the log-value at x: MVN(mean (D,n), cov (D,n,n)) (reference :72-75)."""
        return MultivariateNormal(self.mean_module(x), self._prior_cov(x))

    def sample(self, x, **kwargs):
        return torch.exp(self.forward(x).rsample(**kwargs))

    def conditional_weights(self, xg, ell_g):
        """alpha (D, m) = (K(Xg,Xg) + 1e-4 I)^-1 (log ell_g - c), per dimension: the weights of the conditional mean given
        the lengthscales ell_g (D, m) at the (active columns of the) points xg."""
        xg = self._active(xg)
        c, os, lam = self._hypers()
        eye = torch.eye(xg.shape[0], dtype=xg.dtype, device=xg.device)
        alphas = []
        for b in range(self.input_dim):
            Kgg = F.rbf_ard(xg, xg, lam[b], os[b]) + 1e-4 * eye
            _, P = F.psd_safe_chol_inv(Kgg)
            alphas.append(F.spd_solve(P, torch.log(ell_g[b]) - c[b]))
        return torch.stack(alphas)

    def conditional_sample(self, x, given: Tuple[torch.Tensor, torch.Tensor], **kwargs):
        """exp(c + K(x, Xg) (K(Xg,Xg) + 1e-4 I)^-1 (log ell_g - c))  (reference :80-100) -> (D, n)."""
        xg, ell_g = given
        alpha = self.conditional_weights(xg, ell_g).unsqueeze(-1)  # (D, m, 1)
        x, xg = self._active(x), self._active(xg)
        c, os, lam = self._hypers()
        out = F.rbf_matvec(x.contiguous(), xg.contiguous(), lam, os, alpha, c, True)
        return out.squeeze(-1)

    def log_prob(self, x_and_logell: Tuple[torch.Tensor, torch.Tensor]):
        """Per-dimension log N(log ell_d; c_d, K_d + 1e-4 I) / n (reference :102-109) -> (D,)."""
        x, log_value = x_and_logell
        n = x.shape[-2]
        cov = self._prior_cov(x) + 1e-4 * torch.eye(n, dtype=x.dtype, device=x.device)
        mu = self.mean_module(x)
        out = torch.stack([F.mvn_log_prob(log_value[b], mu[b], cov[b]) for b in range(self.input_dim)])
        return out / n


class GibbsKernel(Kernel):
    """Diagonal Gibbs kernel, R&W eq. 4.32 (reference :111-162).  `forward(x1, x2, ell1, ell2)`; lengthscales (D, n)."""

    is_stationary = False

    def __init__(self, *args, lengthscale_prior: Optional[PositivePriorProcess] = None, **kwargs):
        super().__init__(*args, **kwargs)
        self.lengthscale_prior = lengthscale_prior

    def forward(self, x1, x2, ell1=None, ell2=None, scale=None, **kwargs):
        if ell1 is None:
            ell1 = self.lengthscale_prior.sample(x1)
            self.ell1 = ell1
        if torch.equal(x1, x2):
            ell2 = ell1
        elif ell2 is None:
            ell2 = self.lengthscale_prior.conditional_sample(x2, given=(x1, ell1))
            self.ell2 = ell2
        return F.gibbs_diag(x1, ell1, x2, ell2, scale)


class GibbsSafeScaleKernel(ScaleKernel):
    """Scale wrapper whose batch shape ignores the prior's kernels (reference :164-168).  The outputscale is fused into
    the Gibbs tile kernel when the base kernel is a plain GibbsKernel."""

    def forward(self, x1, x2, diag=False, **params):
        if isinstance(self.base_kernel, GibbsKernel):
            return self.base_kernel.forward(x1, x2, scale=self.outputscale.reshape(1), **params)
        return super().forward(x1, x2, diag=diag, **params)


class InducingGibbsKernel(Kernel):
    """Nystrom / SGPR wrapper for the Gibbs kernel (reference :171-266): `forward(x1, x2, diag=False, ell=...)` with
    `ell` the lengthscales at the inducing points; train / test lengthscales are the conditional mean given them."""

    is_stationary = False

    def __init__(self, base_kernel: GibbsKernel, inducing_points: torch.Tensor, likelihood, active_dims=None):
        super().__init__(active_dims=active_dims)
        self.base_kernel, self.likelihood = base_kernel, likelihood
        if inducing_points.dim() == 1:
            inducing_points = inducing_points.unsqueeze(-1)
        self.register_parameter("inducing_points", torch.nn.Parameter(inducing_points.clone()))

    def _z(self):
        return self.inducing_points

    def _clear_cache(self):
        for a in ("_cached_kernel_mat", "_cached_kernel_inv_root"):
            if hasattr(self, a):
                delattr(self, a)

    def train(self, mode=True):
        self._clear_cache()
        return super().train(mode)

    def _inducing_mat(self, ell=None):
        if not self.training and hasattr(self, "_cached_kernel_mat"):
            return self._cached_kernel_mat
        z = self._z()
        res = self.base_kernel.forward(z, z, ell1=ell)
        if not self.training:
            self._cached_kernel_mat = res
        return res

    def _inducing_inv_root(self, ell=None):
        """U^-1 with Kzz = U^T U (reference :197-208); here U^-1 = (L^-1)^T from the blocked Cholesky + inverse."""
        if not self.training and hasattr(self, "_cached_kernel_inv_root"):
            return self._cached_kernel_inv_root
        _, P = F.psd_safe_chol_inv(self._inducing_mat(ell))
        res = P.T
        if not self.training:
            self._cached_kernel_inv_root = res
        return res

    def _get_covariance(self, x1, x2, ell):
        z = self._z()
        prior = self.base_kernel.lengthscale_prior
        same = torch.equal(x1, x2)
        if same:
            ell1 = prior.conditional_sample(x1, given=(z, ell))
            ell2 = ell1
        else:
            ell_cond = prior.conditional_sample(torch.cat((x1, x2), dim=-2), given=(z, ell))
            ell1, ell2 = ell_cond[..., :x1.shape[-2]], ell_cond[..., x1.shape[-2]:]
        inv_root = self._inducing_inv_root(ell)
        k_ux1 = self.base_kernel.forward(x1, z, ell1=ell1, ell2=ell)
        root1 = F.matmul(k_ux1, inv_root)
        if same:
            covar = LowRankRootCovar(root1)
            if not self.training:
                # SGPR diagonal correction clamp(k_ii - q_ii, 0); k_ii == 1 analytically when ell1 == ell2 (the reference
                # builds a full n x n Gibbs matrix to read this diagonal, gibbs_kernels.py:230)
                corr = (1.0 - covar.diag()).clamp(0, math.inf)
                covar = LowRankRootCovar(root1, corr)
        else:
            k_ux2 = self.base_kernel.forward(x2, z, ell1=ell2, ell2=ell)
            covar = F.matmul(root1, F.matmul(k_ux2, inv_root).T)
        return covar, ell1, ell2

    def forward(self, x1, x2, diag=False, ell=None, **kwargs):
        covar, ell1, ell2 = self._get_covariance(x1, x2, ell=ell)
        if self.training:
            if not torch.equal(x1, x2):
                raise RuntimeError("x1 should equal x2 in training mode")
            prior_diag = torch.ones(x1.shape[-2], dtype=x1.dtype, device=x1.device)  # diag of the unscaled Gibbs kernel
            self.update_added_loss_term("inducing_point_loss_term",
                                        InducingPointKernelAddedLossTerm(prior_diag, covar.diag(), self.likelihood))
        if diag:
            return covar.diag() if isinstance(covar, LowRankRootCovar) else torch.diagonal(covar)
        return covar


class InducingGibbsKernelST(InducingGibbsKernel):
    """Spatio-temporal variant (reference :268-363): identical except that the inducing points are sliced by
    `active_dims` by hand, because ScaleKernel.forward bypasses the base kernel's `__call__`."""

    def _z(self):
        return self.inducing_points[:, self.active_dims]
