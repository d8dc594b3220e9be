"""Torch-facing wrappers of the npgp C ABI: raw launchers (no autograd) and ``torch.autograd.Function``s whose backward
is the hand-written analytic kernel, not an autograd graph.  Every function enqueues on the current CUDA stream and
returns without synchronising."""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import check, lib, ptr, stream


def _c(t: Optional[torch.Tensor]):
    return None if t is None else t.contiguous()


def sym_pack(S: torch.Tensor) -> torch.Tensor:
    """(n,d,d) symmetric -> (n, d(d+1)/2) row-wise upper triangle."""
    d = S.shape[-1]
    iu = torch.triu_indices(d, d, device=S.device)
    return S[..., iu[0], iu[1]].contiguous()


def sym_unpack(Sp: torch.Tensor, d: int) -> torch.Tensor:
    iu = torch.triu_indices(d, d, device=Sp.device)
    S = Sp.new_zeros(*Sp.shape[:-1], d, d)
    S[..., iu[0], iu[1]] = Sp
    S[..., iu[1], iu[0]] = Sp
    return S


# ----------------------------------------------------------------------------------------------------------------------
# raw launchers
# ----------------------------------------------------------------------------------------------------------------------
def gibbs_diag_fwd(x1, ell1, x2, ell2, scale=None, u=None, out=None):
    """K = scale * GibbsKernel(x1, x2; ell1, ell2).  x (n,D), ell (D,n).  Returns K or (K, K@u)."""
    x1, ell1, x2, ell2, scale, u = map(_c, (x1, ell1, x2, ell2, scale, u))
    n1, D = x1.shape
    n2 = x2.shape[0]
    assert ell1.shape == (D, n1) and ell2.shape == (D, n2), "lengthscales must be (D, n)"
    K = out if out is not None else torch.empty(n1, n2, dtype=torch.float64, device=x1.device)
    Ku = torch.zeros(n1, dtype=torch.float64, device=x1.device) if u is not None else None
    check(lib().npgp_gibbs_diag_fwd(D, n1, n2, ptr(x1), ptr(ell1), ptr(x2), ptr(ell2), ptr(scale), ptr(K), K.stride(0),
                                    ptr(u), ptr(Ku), stream()), "npgp_gibbs_diag_fwd")
    return K if u is None else (K, Ku)


def gibbs_diag_bwd(x1, ell1, x2, ell2, scale=None, G=None, rowscale=None, rowvec=None, colvec=None, need_dx1=False,
                   need_dx2=False, need_dscale=False):
    x1, ell1, x2, ell2, scale, G, rowscale, rowvec, colvec = map(
        _c, (x1, ell1, x2, ell2, scale, G, rowscale, rowvec, colvec))
    n1, D = x1.shape
    n2 = x2.shape[0]
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=x1.device)
    d_ell1, d_ell2 = z(D, n1), z(D, n2)
    d_x1 = z(n1, D) if need_dx1 else None
    d_x2 = z(n2, D) if need_dx2 else None
    d_scale = z(()) if need_dscale else None
    check(lib().npgp_gibbs_diag_bwd(D, n1, n2, ptr(x1), ptr(ell1), ptr(x2), ptr(ell2), ptr(scale), ptr(G),
                                    G.stride(0) if G is not None else 0, ptr(rowscale), ptr(rowvec), ptr(colvec),
                                    ptr(d_ell1), ptr(d_x1), ptr(d_ell2), ptr(d_x2), ptr(d_scale), stream()),
          "npgp_gibbs_diag_bwd")
    return dict(d_ell1=d_ell1, d_ell2=d_ell2, d_x1=d_x1, d_x2=d_x2, d_scale=d_scale)


def gibbs_full_fwd(x1, S1p, x2, S2p, jitter=1e-5, scale=None, u=None, out=None):
    """K = scale * full-matrix Gibbs kernel; S?p packed symmetric (n, d(d+1)/2)."""
    x1, S1p, x2, S2p, scale, u = map(_c, (x1, S1p, x2, S2p, scale, u))
    n1, d = x1.shape
    n2 = x2.shape[0]
    P = d * (d + 1) // 2
    assert S1p.shape == (n1, P) and S2p.shape == (n2, P)
    K = out if out is not None else torch.empty(n1, n2, dtype=torch.float64, device=x1.device)
    Ku = torch.zeros(n1, dtype=torch.float64, device=x1.device) if u is not None else None
    check(lib().npgp_gibbs_full_fwd(d, n1, n2, ptr(x1), ptr(S1p), ptr(x2), ptr(S2p), float(jitter), ptr(scale), ptr(K),
                                    K.stride(0), ptr(u), ptr(Ku), stream()), "npgp_gibbs_full_fwd")
    return K if u is None else (K, Ku)


def gibbs_full_bwd(x1, S1p, x2, S2p, jitter=1e-5, scale=None, G=None, rowscale=None, rowvec=None, colvec=None,
                   need_dx1=False, need_dx2=False, need_dscale=False):
    x1, S1p, x2, S2p, scale, G, rowscale, rowvec, colvec = map(
        _c, (x1, S1p, x2, S2p, scale, G, rowscale, rowvec, colvec))
    n1, d = x1.shape
    n2 = x2.shape[0]
    P = d * (d + 1) // 2
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=x1.device)
    d_S1, d_S2 = z(n1, P), z(n2, P)
    d_x1 = z(n1, d) if need_dx1 else None
    d_x2 = z(n2, d) if need_dx2 else None
    d_scale = z(()) if need_dscale else None
    check(lib().npgp_gibbs_full_bwd(d, n1, n2, ptr(x1), ptr(S1p), ptr(x2), ptr(S2p), float(jitter), ptr(scale), ptr(G),
                                    G.stride(0) if G is not None else 0, ptr(rowscale), ptr(rowvec), ptr(colvec),
                                    ptr(d_S1), ptr(d_x1), ptr(d_S2), ptr(d_x2), ptr(d_scale), stream()),
          "npgp_gibbs_full_bwd")
    return dict(d_S1=d_S1, d_S2=d_S2, d_x1=d_x1, d_x2=d_x2, d_scale=d_scale)


def sigma_from_h_fwd(H, Dm):
    H, Dm = _c(H), _c(Dm)
    n, d = H.shape
    S = torch.empty(n, d * (d + 1) // 2, dtype=torch.float64, device=H.device)
    check(lib().npgp_sigma_from_h_fwd(d, n, ptr(H), ptr(Dm), ptr(S), stream()), "npgp_sigma_from_h_fwd")
    return S


def sigma_from_h_bwd(H, Dm, dS, need_dD=True):
    H, Dm, dS = _c(H), _c(Dm), _c(dS)
    n, d = H.shape
    dH = torch.zeros_like(H)
    dD = torch.zeros_like(Dm) if need_dD else None
    check(lib().npgp_sigma_from_h_bwd(d, n, ptr(H), ptr(Dm), ptr(dS), ptr(dH), ptr(dD), stream()),
          "npgp_sigma_from_h_bwd")
    return dH, dD


def rbf_matvec_fwd(x, z, lam, os, V, bias=None, apply_exp=False, out=None):
    """out[b,i,c] = f(bias_b + sum_j os_b exp(-0.5|(x_i-z_j)/lam_b|^2) V[b,j,c]);  lam (nb,d), V (nb,m,nv)."""
    x, z, lam, os, V, bias = map(_c, (x, z, lam, os, V, bias))
    n, d = x.shape
    nb, m, nv = V.shape
    assert lam.shape == (nb, d)
    if out is None:
        out = torch.empty(nb, n, nv, dtype=torch.float64, device=x.device)
    assert out.shape == (nb, n, nv) and out.is_contiguous()
    check(lib().npgp_rbf_matvec_fwd(d, nb, nv, n, m, ptr(x), ptr(z), ptr(lam), ptr(os), ptr(V), ptr(bias),
                                    int(apply_exp), ptr(out), stream()), "npgp_rbf_matvec_fwd")
    return out


def rbf_matvec_bwd(x, z, lam, os, V, dOut, need_dz=True):
    x, z, lam, os, V, dOut = map(_c, (x, z, lam, os, V, dOut))
    n, d = x.shape
    nb, m, nv = V.shape
    dV = torch.zeros_like(V)
    dz = torch.zeros_like(z) if need_dz else None
    check(lib().npgp_rbf_matvec_bwd(d, nb, nv, n, m, ptr(x), ptr(z), ptr(lam), ptr(os), ptr(V), ptr(dOut), ptr(dV),
                                    ptr(dz), stream()), "npgp_rbf_matvec_bwd")
    return dV, dz


def dgemm(A, B, transA=False, transB=False, alpha=1.0, beta=0.0, C=None, tri_a=0, tri_b=0, out_tri=0):
    """C = alpha op(A) op(B) + beta C on the FP64 tensor pipe.  A, B may be views with unit inner stride."""
    assert A.stride(-1) == 1 and B.stride(-1) == 1
    M = A.shape[1] if transA else A.shape[0]
    Kd = A.shape[0] if transA else A.shape[1]
    N = B.shape[0] if transB else B.shape[1]
    assert (B.shape[1] if transB else B.shape[0]) == Kd
    if C is None:
        C = torch.empty(M, N, dtype=torch.float64, device=A.device)
        assert beta == 0.0
    check(lib().npgp_dgemm(int(transA), int(transB), M, N, Kd, float(alpha), ptr(A), A.stride(0), ptr(B), B.stride(0),
                           float(beta), ptr(C), C.stride(0), tri_a, tri_b, out_tri, stream()), "npgp_dgemm")
    return C


def rowquad(K, Cm, need_q=True, T=None):
    """T = K @ Cm, q_i = sum_j T_ij K_ij."""
    n, M = K.shape
    if T is None:
        T = torch.empty(n, M, dtype=torch.float64, device=K.device)
    q = torch.zeros(n, dtype=torch.float64, device=K.device) if need_q else None
    check(lib().npgp_rowquad(n, M, ptr(K), K.stride(0), ptr(Cm), Cm.stride(0), ptr(T), T.stride(0), ptr(q), stream()),
          "npgp_rowquad")
    return T, q


# ----------------------------------------------------------------------------------------------------------------------
# exact int8 tensor-core contractions (csrc/oz8.cu).  Workspaces are owned by the CALLER (an I8Workspace per model / call
# site): nothing here is process-global, so two models or two streams never share scratch memory.
# ----------------------------------------------------------------------------------------------------------------------
class I8Workspace:
    """Scratch memory of the int8 contractions for one call site, keyed by shape.  Buffers are created on first use (do that
    before CUDA-graph capture) and live as long as this object, so a captured graph that holds raw pointers into them
    stays valid for the life of the model that owns the workspace."""

    def __init__(self):
        self._bufs = {}

    def get(self, key, nbytes, device, dtype=torch.uint8):
        buf = self._bufs.get(key)
        item = torch.empty((), dtype=dtype).element_size()
        if buf is None or buf.numel() * item < nbytes or buf.device != device:
            buf = self._bufs[key] = torch.empty((nbytes + item - 1) // item, dtype=dtype, device=device)
        return buf


_DEFAULT_I8_WS = {}  # one workspace per (device, stream) for callers that do not pass their own


def _ws(workspace, device):
    if workspace is not None:
        return workspace
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    if key not in _DEFAULT_I8_WS:
        _DEFAULT_I8_WS[key] = I8Workspace()
    return _DEFAULT_I8_WS[key]


def rowquad_i8(K, Cm, need_q=True, T=None, workspace=None):
    """rowquad on the integer tensor cores (tcgen05 kind::i8, exact byte-digit split, see csrc/oz8.cu).  Cm must be
    symmetric and M a multiple of 64."""
    n, M = K.shape
    if T is None:
        T = torch.empty(n, M, dtype=torch.float64, device=K.device)
    q = torch.zeros(n, dtype=torch.float64, device=K.device) if need_q else None
    nbytes = lib().npgp_rowquad_i8_workspace_bytes(n, M)
    work = _ws(workspace, K.device).get(("rowquad", n, M), nbytes, K.device)
    check(lib().npgp_rowquad_i8(n, M, ptr(K), K.stride(0), ptr(Cm), Cm.stride(0), ptr(T), T.stride(0), ptr(q), ptr(work),
                                nbytes, stream()), "npgp_rowquad_i8")
    return T, q


def _syrk_i8_work(K, workspace):
    n, M = K.shape
    nbytes = lib().npgp_syrk_i8_workspace_bytes(n, M)
    return _ws(workspace, K.device).get(("syrk", n, M), nbytes, K.device), nbytes


def syrk_i8(K, w0=None, alpha=1.0, out=None, workspace=None):
    """alpha * w0 * K^T K (symmetric M x M) on the integer tensor cores (exact byte-digit split, csrc/oz8.cu); w0: device
    scalar (or None); M must be a multiple of 128.  Bitwise reproducible (chunk partials are added in a fixed order)."""
    n, M = K.shape
    if out is None:
        out = torch.empty(M, M, dtype=torch.float64, device=K.device)
    work, nbytes = _syrk_i8_work(K, workspace)
    check(lib().npgp_syrk_i8(n, M, float(alpha), ptr(K), K.stride(0), ptr(w0), None, 0.0, 0, ptr(out), out.stride(0),
                             ptr(work), nbytes, stream()), "npgp_syrk_i8")
    return out


def wsyrk_i8(K, w, uniform_count, uniform_target, alpha=1.0, out=None, workspace=None):
    """alpha * K^T diag(w) K with the device-side equal-weights gate of `wsyrk`: equal weights run on the integer tensor
    cores, unequal ones on the FP64 weighted kernel; both are enqueued and the one the flag does not select exits at once."""
    n, M = K.shape
    if out is None:
        out = torch.empty(M, M, dtype=torch.float64, device=K.device)
    w = _c(w)
    check(lib().npgp_wsyrk_weighted_only(n, M, float(alpha), ptr(K), K.stride(0), ptr(w), ptr(uniform_count),
                                         float(uniform_target), ptr(out), out.stride(0), stream()),
          "npgp_wsyrk_weighted_only")
    work, nbytes = _syrk_i8_work(K, workspace)
    check(lib().npgp_syrk_i8(n, M, float(alpha), ptr(K), K.stride(0), ptr(w), ptr(uniform_count), float(uniform_target), 1,
                             ptr(out), out.stride(0), ptr(work), nbytes, stream()), "npgp_syrk_i8")
    return out


# ---- digit-plane path: K(X,Z) exists only as 7 bytes per entry -------------------------------------------------------
def digits_bytes(rows, Kd, block_rows=128):
    return lib().npgp_o8_digits_bytes(rows, Kd, block_rows)


def gibbs_digits_splits(n1, n2):
    return lib().npgp_gibbs_digits_splits(n1, n2)


def gibbs_diag_fwd_digits(x1, ell1, x2, ell2, scale, digits, u=None, Ku_part=None):
    """Digit planes of scale * GibbsKernel(x1, x2) (row layout, see csrc/oz8.cuh) into `digits` (uint8); with u the partial
    sums of K u go to Ku_part (splits, n1)."""
    x1, ell1, x2, ell2, scale, u = map(_c, (x1, ell1, x2, ell2, scale, u))
    n1, D = x1.shape
    n2 = x2.shape[0]
    check(lib().npgp_gibbs_diag_fwd_digits(D, n1, n2, ptr(x1), ptr(ell1), ptr(x2), ptr(ell2), ptr(scale), ptr(digits), ptr(u),
                                           ptr(Ku_part), Ku_part.stride(0) if Ku_part is not None else 0, stream()),
          "npgp_gibbs_diag_fwd_digits")
    return digits


def gibbs_full_fwd_digits(x1, S1p, x2, S2p, jitter, scale, digits, u=None, Ku_part=None):
    x1, S1p, x2, S2p, scale, u = map(_c, (x1, S1p, x2, S2p, scale, u))
    n1, d = x1.shape
    n2 = x2.shape[0]
    check(lib().npgp_gibbs_full_fwd_digits(d, n1, n2, ptr(x1), ptr(S1p), ptr(x2), ptr(S2p), float(jitter), ptr(scale),
                                           ptr(digits), ptr(u), ptr(Ku_part),
                                           Ku_part.stride(0) if Ku_part is not None else 0, stream()),
          "npgp_gibbs_full_fwd_digits")
    return digits


def o8_slice_rows(X, block_rows, digits, expo):
    """Digit planes + per-row exponents of an arbitrary FP64 matrix (block_rows 128: A operand, 64: symmetric B operand)."""
    R, Kd = X.shape
    check(lib().npgp_o8_slice_rows(R, Kd, ptr(X), X.stride(0), block_rows, ptr(digits), ptr(expo), stream()),
          "npgp_o8_slice_rows")


def o8_rowquad_digits(n, M, a_digits, a_scale, c_digits, c_expo, T, q_part=None, gvec=None, du_part=None, a_expo=None,
                      Kmat=None):
    """T = K C from digit planes; q_part (M/64, n) receives the per-column-block partials of rowdot(T, K); du_part
    (ceil(n/128), M) the per-row-block partials of K^T gvec.  a_scale: device scalar bounding the entries of K (matrix-wide
    exponent) unless per-row exponents a_expo are given.  T = None (with q_part): the row dot only, T is not stored."""
    check(lib().npgp_o8_rowquad_digits(n, M, ptr(a_digits), ptr(a_expo), ptr(a_scale), ptr(c_digits), ptr(c_expo), ptr(Kmat),
                                       Kmat.stride(0) if Kmat is not None else 0, ptr(T), T.stride(0) if T is not None else M,
                                       ptr(q_part), q_part.stride(0) if q_part is not None else 0, ptr(gvec), ptr(du_part),
                                       stream()),
          "npgp_o8_rowquad_digits")
    return T


def o8_sum_partials(part, out=None):
    nb, N = part.shape
    if out is None:
        out = torch.empty(N, dtype=torch.float64, device=part.device)
    check(lib().npgp_o8_sum_partials(nb, N, ptr(part), ptr(out), stream()), "npgp_o8_sum_partials")
    return out


def o8_trinorm_digits(n, N, Kd, a_digits, a_scale, b_digits, b_expo, q_part, Ms=0, a_expo=None):
    """q_part[cb, i] = sum_{j in column block cb} (A B^T)_ij^2 with B (N x Kd) lower triangular (block diagonal with its split
    at column Ms when Ms > 0); q_part (N/64, >= n).  a_scale: device scalar bounding A unless per-row exponents a_expo."""
    check(lib().npgp_o8_trinorm_digits(n, N, Kd, Ms, ptr(a_digits), ptr(a_expo), ptr(a_scale), ptr(b_digits), ptr(b_expo),
                                       ptr(q_part), q_part.stride(0), stream()), "npgp_o8_trinorm_digits")
    return q_part


def o8_gemm_digits(n, N, Kd, a_digits, a_scale, b_digits, b_expo, T, a_expo=None):
    """T (n x N) = A B^T from planes, stored only: A (n x Kd, block_rows 128), B (N x Kd, block_rows 64, per-row exponents
    b_expo).  a_scale: device scalar bounding A unless per-row exponents a_expo.  T: row stride even and >= N."""
    check(lib().npgp_o8_gemm_digits(n, N, Kd, ptr(a_digits), ptr(a_expo), ptr(a_scale), ptr(b_digits), ptr(b_expo), ptr(T),
                                    T.stride(0), stream()), "npgp_o8_gemm_digits")
    return T


def sample_normals(W, S, seed, Et):
    """Et (Sp, W) = E^T of S draws: Et[s, j] = normal_from_index(seed, (s << 32) + j) for s < S, zero rows s >= S."""
    assert Et.shape[1] == W and Et.is_contiguous()
    check(lib().npgp_sample_normals(W, S, Et.shape[0], int(seed), ptr(Et), stream()), "npgp_sample_normals")
    return Et


def sgpr_sample_finish(mean, qn, nb_t, F, S, s, noise, out, os_t=None, add_noise=False, seed=0, row0=0):
    """Draws of one chunk: out[s, i] = mean_i + F[i, s] + sqrt(r_i (+ noise)) xi_s(row0 + i) for s < S, with the residual r
    of the row-norm partials qn (nb_t temporal blocks, then the Gibbs ones); out may be a column view (row stride >= n)."""
    n = mean.shape[0]
    assert F.stride(1) == 1 and out.stride(1) == 1
    check(lib().npgp_sgpr_sample_finish(n, S, ptr(mean), ptr(qn), qn.stride(0), nb_t, qn.shape[0] - nb_t, ptr(F), F.stride(0),
                                        ptr(s), ptr(noise), ptr(os_t), int(bool(add_noise)), int(seed), int(row0), ptr(out),
                                        out.stride(0), stream()), "npgp_sgpr_sample_finish")
    return out


def sgpr_rownorm_parts(G, q_part):
    """q_part[cb, i] = sum_{j in [64 cb, 64 cb + 64)} G_ij^2 (FP64; G may be a column view)."""
    n, W = G.shape
    assert G.stride(1) == 1
    check(lib().npgp_sgpr_rownorm_parts(n, W, ptr(G), G.stride(0), ptr(q_part), q_part.stride(0), stream()),
          "npgp_sgpr_rownorm_parts")
    return q_part


def sgpr_predict_workspace(n, device):
    """Zeroed workspace of sgpr_predict_finish for chunks of up to n rows (its ticket must start at 0)."""
    return torch.zeros(lib().npgp_sgpr_predict_workspace_bytes(n), dtype=torch.uint8, device=device)


def sgpr_predict_finish(qn, nb_t, qv, s, noise, var_f, os_t=None, mean=None, y=None, var_y=None, lpd=None, sums=None,
                        work=None):
    """Predictive variances (and with y: lpd, accumulated sums) of one chunk from the row-norm partials qn (nb_t temporal
    blocks, then the Gibbs ones) and qv; see npgp_sgpr_predict_finish."""
    n = var_f.shape[0]
    nbn, nbv = qn.shape[0], qv.shape[0]
    nbytes = work.numel() if work is not None else 0
    check(lib().npgp_sgpr_predict_finish(n, ptr(qn), qn.stride(0), nb_t, nbn - nb_t, ptr(qv), qv.stride(0), nbv, ptr(mean),
                                         ptr(y), ptr(s), ptr(noise), ptr(os_t), ptr(var_f), ptr(var_y), ptr(lpd), ptr(sums),
                                         ptr(work), nbytes, stream()), "npgp_sgpr_predict_finish")
    return var_f


def exact_predict_finish(qn, s, noise, add_var, var_f, mean=None, y=None, var_y=None, lpd=None, sums=None, work=None):
    """The exact GP's predictive variances (and with y: lpd, accumulated sums) of one chunk from the partials qn of
    |P_y k|^2: var_f = s max(1 - q, 0) + add_var; see npgp_exact_predict_finish."""
    n = var_f.shape[0]
    nbytes = work.numel() if work is not None else 0
    check(lib().npgp_exact_predict_finish(n, ptr(qn), qn.stride(0), qn.shape[0], ptr(mean), ptr(y), ptr(s), ptr(noise),
                                          float(add_var), ptr(var_f), ptr(var_y), ptr(lpd), ptr(sums), ptr(work), nbytes,
                                          stream()), "npgp_exact_predict_finish")
    return var_f


def o8_syrk_part_bytes(n, M):
    return lib().npgp_o8_syrk_part_bytes(n, M)


def o8_syrk_digits(n, M, digits, scale, part, w0=None, alpha=1.0, skip_count=None, skip_rows=None, out=None,
                   accumulate=False):
    """alpha * w0 * (K^T K - sum_{i in skip} k_i k_i^T) from the row-layout digit planes of K (read MN-major)."""
    if out is None:
        out = torch.empty(M, M, dtype=torch.float64, device=digits.device)
    nbytes = part.numel() * part.element_size()
    check(lib().npgp_o8_syrk_digits(n, M, ptr(digits), ptr(scale), float(alpha), ptr(w0), ptr(skip_count), ptr(skip_rows),
                                    int(accumulate), ptr(out), out.stride(0), ptr(part), nbytes, stream()),
          "npgp_o8_syrk_digits")
    return out


def mu_gmu_parts(y, mu_part, noise, wscale):
    """mu = sum of the partial mean vectors (rows of mu_part), gmu = wscale (y - mu) / noise."""
    nparts, n = mu_part.shape
    mu = torch.empty(n, dtype=torch.float64, device=y.device)
    gmu = torch.empty_like(mu)
    check(lib().npgp_mu_gmu_parts(n, ptr(_c(y)), ptr(mu_part), nparts, mu_part.stride(0), ptr(noise), float(wscale), ptr(mu),
                                  ptr(gmu), stream()), "npgp_mu_gmu_parts")
    return mu, gmu


def gauss_ell_parts(y, mu, q_part, kdiag, noise, jitter_xx=1e-4, min_var=1e-6, wscale=1.0, want_var=False,
                    skip_count=None, skip_rows=None):
    """Deterministic gauss_ell with q = sum of the rows of q_part.  Returns (acc4, gmu, gv, var); acc4[3] is the weight
    w0 = -0.5 wscale / noise of every unclamped row; clamped rows are appended to skip_rows."""
    n = y.shape[0]
    z = lambda *s: torch.empty(*s, dtype=torch.float64, device=y.device)
    gmu, gv = z(n), z(n)
    var = z(n) if want_var else None
    acc = z(4)
    nbytes = lib().npgp_gauss_ell_parts_workspace_bytes(n)
    work = z(nbytes // 8 + 1)
    nq = q_part.shape[0] if q_part is not None else 0
    check(lib().npgp_gauss_ell_parts(n, ptr(_c(y)), ptr(mu), ptr(q_part), nq, q_part.stride(0) if nq else 0, ptr(kdiag),
                                     float(jitter_xx), float(min_var), ptr(noise), float(wscale), ptr(var), ptr(gmu), ptr(gv),
                                     ptr(acc), ptr(skip_count), ptr(skip_rows), ptr(work), nbytes, stream()),
          "npgp_gauss_ell_parts")
    return acc, gmu, gv, var


def wsyrk(K, w=None, alpha=1.0, out=None, uniform_count=None, uniform_target=0.0):
    """alpha * K^T diag(w) K (symmetric M x M).  uniform_count (device scalar) == uniform_target tells the kernel, on
    the device, that all weights are equal."""
    n, M = K.shape
    if out is None:
        out = torch.empty(M, M, dtype=torch.float64, device=K.device)
    if uniform_count is not None and w is not None:
        check(lib().npgp_wsyrk_hint(n, M, float(alpha), ptr(K), K.stride(0), ptr(_c(w)), ptr(uniform_count),
                                    float(uniform_target), ptr(out), out.stride(0), stream()), "npgp_wsyrk_hint")
    else:
        check(lib().npgp_wsyrk(n, M, float(alpha), ptr(K), K.stride(0), ptr(_c(w)), ptr(out), out.stride(0), stream()),
              "npgp_wsyrk")
    return out


POTRF_IMPL = "flow"  # "flow": one dataflow kernel (csrc/chol_flow.cu); "steps": one kernel per panel step (csrc/chol.cu)


def potrf_inv(A, overwrite=False, impl=None):
    """Lower Cholesky factor L of A and P = L^-1.  Returns (L, P, info) with info a device int32 scalar
    (0 = ok, > 0: 1-based index of the first non-positive pivot, -1: dataflow wait timed out)."""
    M = A.shape[0]
    L = A if overwrite else A.clone()
    assert L.is_contiguous()
    P = torch.empty_like(L)
    info = torch.zeros((), dtype=torch.int32, device=A.device)
    if (impl or POTRF_IMPL) == "flow":
        nbytes = lib().npgp_potrf_flow_workspace_bytes(M)
        work = torch.empty(nbytes // 4 + 1, dtype=torch.int32, device=A.device)
        check(lib().npgp_potrf_inv_flow(M, ptr(L), L.stride(0), ptr(P), P.stride(0), ptr(work), nbytes, ptr(info),
                                        stream()), "npgp_potrf_inv_flow")
        return L, P, info
    nbytes = lib().npgp_potrf_workspace_bytes(M)
    work = torch.empty(nbytes // 8 + 1, dtype=torch.float64, device=A.device)
    check(lib().npgp_potrf_inv_lower(M, ptr(L), L.stride(0), ptr(P), P.stride(0), ptr(work), nbytes, ptr(info),
                                     stream()), "npgp_potrf_inv_lower")
    return L, P, info


def potrf_inv_batch(mats):
    """Lower Cholesky factors and inverse factors of up to 4 SPD matrices of the same order in ONE dataflow launch
    (npgp_potrf_inv_flow_batch).  Returns [(L, P, info), ...]; the inputs are not modified."""
    import ctypes as C
    n, M = len(mats), mats[0].shape[0]
    Ls = [A.clone() for A in mats]
    Ps = [torch.empty_like(A) for A in mats]
    infos = [torch.zeros((), dtype=torch.int32, device=mats[0].device) for _ in mats]
    nbytes = lib().npgp_potrf_flow_workspace_bytes(M)
    works = [torch.empty(nbytes // 4 + 1, dtype=torch.int32, device=mats[0].device) for _ in mats]
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    check(lib().npgp_potrf_inv_flow_batch(n, M, arr(Ls), Ls[0].stride(0), arr(Ps), Ps[0].stride(0), arr(works), nbytes,
                                          arr(infos), stream()), "npgp_potrf_inv_flow_batch")
    return list(zip(Ls, Ps, infos))


def colwsum(K, w=None, out=None):
    """out[j] (+)= sum_i w_i K[i,j]."""
    n, M = K.shape
    if out is None:
        out = torch.zeros(M, dtype=torch.float64, device=K.device)
    check(lib().npgp_colwsum(n, M, ptr(K), K.stride(0), ptr(_c(w)), ptr(out), stream()), "npgp_colwsum")
    return out


def _segsum_work(n, R, full, device):
    nbytes = lib().npgp_segsum_workspace_bytes(n, R, int(full))
    if nbytes < 0:
        raise ValueError("no pair-sum workspace for n = %d rows, R = %d regions" % (n, R))
    work = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
    return work, work.data_ptr() + (-work.data_ptr()) % 256, nbytes


def gibbs_diag_segsum(x, ell, seg, w=None, full=False, part=0, nparts=1, scale=None):
    """Pair sums G[r, r'] = scale * sum_{i in r, j in r'} w_i w_j kappa(x_i, x_j) of the diagonal Gibbs kernel over the regions
    rows [seg[r], seg[r+1]) (int64, R + 1 offsets).  x (n,D), ell (D,n).  Returns (Gdiag (R), G (R,R) or None)."""
    x, ell, w, scale, seg = map(_c, (x, ell, w, scale, seg))
    n, D = x.shape
    R = seg.numel() - 1
    f64 = dict(dtype=torch.float64, device=x.device)
    Gdiag = torch.empty(R, **f64)
    G = torch.empty(R, R, **f64) if full else None
    _, wp, nbytes = work = _segsum_work(n, R, full, x.device)
    check(lib().npgp_gibbs_diag_segsum(D, n, ptr(x), ptr(ell), ptr(w), R, ptr(seg), int(full), part, nparts, ptr(scale),
                                       ptr(Gdiag), ptr(G), R, wp, nbytes, stream()), "npgp_gibbs_diag_segsum")
    return Gdiag, G


def gibbs_full_segsum(x, S1p, seg, w=None, jitter=1e-5, full=False, part=0, nparts=1, scale=None):
    """The same for the full-matrix Gibbs kernel: S1p (n, d(d+1)/2) packed, jitter as gibbs_full_fwd."""
    x, S1p, w, scale, seg = map(_c, (x, S1p, w, scale, seg))
    n, d = x.shape
    R = seg.numel() - 1
    f64 = dict(dtype=torch.float64, device=x.device)
    Gdiag = torch.empty(R, **f64)
    G = torch.empty(R, R, **f64) if full else None
    _, wp, nbytes = work = _segsum_work(n, R, full, x.device)
    check(lib().npgp_gibbs_full_segsum(d, n, ptr(x), ptr(S1p), float(jitter), ptr(w), R, ptr(seg), int(full), part, nparts,
                                       ptr(scale), ptr(Gdiag), ptr(G), R, wp, nbytes, stream()), "npgp_gibbs_full_segsum")
    return Gdiag, G


def segment_colwsum(K, seg, w=None, row0=0, out=None):
    """out[r, j] (+)= sum_{i in r} w_i K[i - row0, j] for the rows row0 .. row0 + n - 1 of the sorted set (seg: R + 1 offsets)."""
    n, M = K.shape
    seg, w = _c(seg), _c(w)
    R = seg.numel() - 1
    if out is None:
        out = torch.zeros(R, M, dtype=torch.float64, device=K.device)
    nbytes = lib().npgp_segment_colwsum_workspace_bytes(n, M)
    work = torch.empty(max(nbytes, 8) // 8, dtype=torch.float64, device=K.device)
    check(lib().npgp_segment_colwsum(n, M, ptr(K), K.stride(0), ptr(w), row0, R, ptr(seg), ptr(out), out.stride(0), ptr(work),
                                     nbytes, stream()), "npgp_segment_colwsum")
    return out


def gemv_n(A, v, out=None):
    """A @ v (one warp per row)."""
    n, M = A.shape
    if out is None:
        out = torch.empty(n, dtype=torch.float64, device=A.device)
    check(lib().npgp_gemv_n(n, M, ptr(A), A.stride(0), ptr(_c(v)), ptr(out), stream()), "npgp_gemv_n")
    return out


def gauss_ell(y, mu, q, kdiag, noise, jitter_xx=1e-4, min_var=1e-6, wscale=1.0, want_var=False):
    """Gaussian expected log-lik sums + gradient seeds; kdiag, noise are device scalars.  Returns (acc3, gmu, gv, var)."""
    n = y.shape[0]
    z = lambda *s: torch.empty(*s, dtype=torch.float64, device=y.device)
    gmu, gv = z(n), z(n)
    var = z(n) if want_var else None
    acc = torch.zeros(3, dtype=torch.float64, device=y.device)
    check(lib().npgp_gauss_ell(n, ptr(_c(y)), ptr(mu), ptr(q), ptr(kdiag), float(jitter_xx), float(min_var), ptr(noise),
                               float(wscale), ptr(var), ptr(gmu), ptr(gv), ptr(acc), stream()), "npgp_gauss_ell")
    return acc, gmu, gv, var


def phi_mask_(X, alpha=1.0):
    check(lib().npgp_phi_mask(X.shape[0], ptr(X), X.stride(0), float(alpha), stream()), "npgp_phi_mask")
    return X


def adam_step_(p, g, m, v, step, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8, gscale=1.0, mask=None):
    check(lib().npgp_adam_step(p.numel(), ptr(p), ptr(g), ptr(m), ptr(v), ptr(mask), float(lr), float(beta1),
                               float(beta2), float(eps), int(step), float(gscale), stream()), "npgp_adam_step")
    return p


def adam_step_dev_(p, g, m, v, step_dev, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8, gscale=1.0, mask=None):
    """Adam with the step counter on the device (graph-capturable)."""
    check(lib().npgp_adam_step_dev(p.numel(), ptr(p), ptr(g), ptr(m), ptr(v), ptr(mask), float(lr), float(beta1),
                                   float(beta2), float(eps), ptr(step_dev), float(gscale), stream()),
          "npgp_adam_step_dev")
    return p


# ----------------------------------------------------------------------------------------------------------------------
# autograd Functions (analytic backward kernels)
# ----------------------------------------------------------------------------------------------------------------------
class GibbsDiagFn(torch.autograd.Function):
    """K = scale * GibbsKernel(x1,x2;ell1,ell2) with gradients to x1, ell1, x2, ell2, scale -- the set the reference
    obtains through autograd (SURVEY Appendix A.4)."""

    @staticmethod
    def forward(ctx, x1, ell1, x2, ell2, scale):
        ctx.save_for_backward(x1, ell1, x2, ell2, scale)
        return gibbs_diag_fwd(x1.detach(), ell1.detach(), x2.detach(), ell2.detach(),
                              None if scale is None else scale.detach())

    @staticmethod
    def backward(ctx, G):
        x1, ell1, x2, ell2, scale = ctx.saved_tensors
        nd = ctx.needs_input_grad
        r = gibbs_diag_bwd(x1, ell1, x2, ell2, scale, G=G, need_dx1=nd[0], need_dx2=nd[2],
                           need_dscale=scale is not None and nd[4])
        return (r["d_x1"], r["d_ell1"] if nd[1] else None, r["d_x2"], r["d_ell2"] if nd[3] else None,
                r["d_scale"].reshape(scale.shape) if (scale is not None and nd[4]) else None)


class GibbsFullFn(torch.autograd.Function):
    """Full-matrix Gibbs kernel from packed Sigma; gradients to x1, S1p, x2, S2p, scale (packed-symmetric convention
    converted so that the returned grad is w.r.t. the PACKED entries: off-diagonals count twice)."""

    @staticmethod
    def forward(ctx, x1, S1p, x2, S2p, scale, jitter):
        ctx.save_for_backward(x1, S1p, x2, S2p, scale)
        ctx.jitter = jitter
        return gibbs_full_fwd(x1.detach(), S1p.detach(), x2.detach(), S2p.detach(), jitter,
                              None if scale is None else scale.detach())

    @staticmethod
    def backward(ctx, G):
        x1, S1p, x2, S2p, scale = ctx.saved_tensors
        nd = ctx.needs_input_grad
        r = gibbs_full_bwd(x1, S1p, x2, S2p, ctx.jitter, scale, G=G, need_dx1=nd[0], need_dx2=nd[2],
                           need_dscale=scale is not None and nd[4])
        d = x1.shape[1]
        mult = _offdiag_multiplier(d, x1.device)
        return (r["d_x1"], r["d_S1"] * mult if nd[1] else None, r["d_x2"], r["d_S2"] * mult if nd[3] else None,
                r["d_scale"].reshape(scale.shape) if (scale is not None and nd[4]) else None, None)


def _offdiag_multiplier(d, device):
    iu = torch.triu_indices(d, d, device=device)
    return torch.where(iu[0] == iu[1], 1.0, 2.0).to(torch.float64)


class SigmaFromHFn(torch.autograd.Function):
    """Packed Sigma(h) (multivariate_gibbs_kernel.py:98).  Incoming grad is w.r.t. packed entries."""

    @staticmethod
    def forward(ctx, H, Dm):
        ctx.save_for_backward(H, Dm)
        return sigma_from_h_fwd(H.detach(), Dm.detach())

    @staticmethod
    def backward(ctx, dSp):
        H, Dm = ctx.saved_tensors
        d = H.shape[1]
        # kernel expects entries of the symmetric-matrix gradient: packed grad / multiplicity
        dH, dD = sigma_from_h_bwd(H, Dm, dSp / _offdiag_multiplier(d, H.device), need_dD=ctx.needs_input_grad[1])
        return dH if ctx.needs_input_grad[0] else None, dD


class RbfMatvecFn(torch.autograd.Function):
    """Matrix-free field interpolation; gradients to z and V (the prior hyper-parameters lam/os/bias are frozen in the
    reference's experiments, spatial_exp.py:166-167, and get no gradient here)."""

    @staticmethod
    def forward(ctx, x, z, lam, os, V, bias, apply_exp):
        out = rbf_matvec_fwd(x.detach(), z.detach(), lam.detach(), None if os is None else os.detach(), V.detach(),
                             None if bias is None else bias.detach(), apply_exp)
        ctx.save_for_backward(x, z, lam, os, V, out if apply_exp else None)
        ctx.apply_exp = apply_exp
        return out

    @staticmethod
    def backward(ctx, dOut):
        x, z, lam, os, V, out = ctx.saved_tensors
        if ctx.apply_exp:
            dOut = dOut * out
        dV, dz = rbf_matvec_bwd(x, z, lam, os, V, dOut, need_dz=ctx.needs_input_grad[1])
        return None, dz, None, None, dV if ctx.needs_input_grad[4] else None, None, None


ROWQUAD_SYM_I8 = True  # rowquad_sym's forward product on the int8 tensor cores when the width allows (DGP layers)


class RowquadFn(torch.autograd.Function):
    """q_i = k_i^T C k_i for SYMMETRIC C (T = K C on the FP64 tensor pipe with the row-dot fused in the epilogue).
    Backward: dK = 2 diag(dq) T,  dC = K^T diag(dq) K (wsyrk)."""

    @staticmethod
    def forward(ctx, K, Cm):
        Kc, Cc = K.detach().contiguous(), Cm.detach().contiguous()
        if ROWQUAD_SYM_I8 and Kc.shape[1] % 64 == 0 and Kc.shape[0] >= 4096:
            # exact byte-digit split on the integer tensor cores (same result to FP64 rounding, ~2.4x the DMMA rate)
            T, q = rowquad_i8(Kc, Cc)
        else:
            T, q = rowquad(Kc, Cc)
        ctx.save_for_backward(Kc, T)
        return q

    @staticmethod
    def backward(ctx, dq):
        K, T = ctx.saved_tensors
        dK = (2.0 * dq).unsqueeze(-1) * T if ctx.needs_input_grad[0] else None
        dC = wsyrk(K, dq.contiguous()) if ctx.needs_input_grad[1] else None
        return dK, dC


class DsviSampleFn(torch.autograd.Function):
    """h = mu + sqrt(var) * eps (DeepGPLayer's Normal(mean, sqrt(variance)).rsample()); eps given or Philox-generated."""

    @staticmethod
    def forward(ctx, mu, var, eps, seed, offset):
        muc, varc = mu.detach().contiguous(), var.detach().contiguous()
        h = torch.empty_like(muc)
        eps_out = torch.empty_like(muc) if eps is None else None
        check(lib().npgp_dsvi_sample(muc.numel(), ptr(muc), ptr(varc), ptr(_c(eps)), int(seed), int(offset), ptr(h),
                                     ptr(eps_out), stream()), "npgp_dsvi_sample")
        ctx.save_for_backward(varc, eps_out if eps is None else _c(eps))
        return h

    @staticmethod
    def backward(ctx, dh):
        var, eps = ctx.saved_tensors
        dh = dh.contiguous()
        dmu, dvar = torch.empty_like(var), torch.empty_like(var)
        check(lib().npgp_dsvi_sample_bwd(var.numel(), ptr(var), ptr(eps), ptr(dh), ptr(dmu), ptr(dvar), stream()),
              "npgp_dsvi_sample_bwd")
        return dmu, dvar, None, None, None


class DsviLayerFn(torch.autograd.Function):
    """(mean = K u, var, info) of one output dimension of a whitened-SVGP deep-GP layer with an RBF-ARD * Scale kernel, forward
    and analytic backward each ONE C call (csrc/dsvi_layer.cu: npgp_dsvi_layer_fwd / _bwd).  K, T = K C and the Z-side factors
    travel from forward to backward in the call's workspace."""

    @staticmethod
    def forward(ctx, X, Z, ls, os, m, Ls, jitter):
        Xc, Zc, lsc, osc, mc, Lsc = (t.detach().contiguous() for t in (X, Z, ls.reshape(-1), os.reshape(1), m, Ls))
        n, d = Xc.shape
        M = Zc.shape[0]
        nbytes = lib().npgp_dsvi_layer_workspace_bytes(n, M, d)
        if nbytes < 0:
            raise _lib.NpgpError("npgp_dsvi_layer: unsupported shape n=%d M=%d d=%d" % (n, M, d))
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=Xc.device)
        off = (-ws.data_ptr()) % 256
        mean = torch.empty(n, dtype=torch.float64, device=Xc.device)
        var = torch.empty_like(mean)
        info = torch.zeros((), dtype=torch.int32, device=Xc.device)
        check(lib().npgp_dsvi_layer_fwd(n, M, d, ptr(Xc), ptr(Zc), ptr(lsc), ptr(osc), ptr(mc), ptr(Lsc), float(jitter), 1e-4, 1e-6,
                                        ptr(mean), ptr(var), ptr(info), ws.data_ptr() + off, nbytes, stream()),
              "npgp_dsvi_layer_fwd")
        ctx.save_for_backward(Xc, Zc, lsc, osc, mc, var)
        ctx.ws, ctx.off, ctx.nbytes, ctx.shapes = ws, off, nbytes, (ls.shape, os.shape)
        ctx.mark_non_differentiable(info)
        return mean, var, info

    @staticmethod
    def backward(ctx, dmean, dvar, _):
        Xc, Zc, lsc, osc, mc, var = ctx.saved_tensors
        n, d = Xc.shape
        M = Zc.shape[0]
        z = lambda *s: torch.empty(*s, dtype=torch.float64, device=Xc.device)
        dmean = dmean.contiguous() if dmean is not None else torch.zeros_like(var)
        dvar = dvar.contiguous() if dvar is not None else torch.zeros_like(var)
        dX = z(n, d) if ctx.needs_input_grad[0] else None
        dZ, dls, dos, dm, dLs = z(M, d), z(d), z(1), z(M), z(M, M)
        check(lib().npgp_dsvi_layer_bwd(n, M, d, ptr(Xc), ptr(Zc), ptr(lsc), ptr(osc), ptr(mc), ptr(var), 1e-6, ptr(dmean),
                                        ptr(dvar), ptr(dX), ptr(dZ), ptr(dls), ptr(dos), ptr(dm), ptr(dLs),
                                        ctx.ws.data_ptr() + ctx.off, ctx.nbytes, stream()), "npgp_dsvi_layer_bwd")
        ctx.ws = None  # K and T (2 x n x M doubles) are released here
        ls_shape, os_shape = ctx.shapes
        return dX, dZ, dls.reshape(ls_shape), dos.reshape(os_shape), dm, dLs, None


def dsvi_layer(X, Z, ls, os, m, Ls, jitter=1e-6):
    return DsviLayerFn.apply(X, Z, ls, os, m, Ls, jitter)


class GaussEllBatchedFn(torch.autograd.Function):
    """sums[s] = sum_i E_q log N(y_i | f_si, noise) for mu, var of shape (S, n); gradients to mu, var and noise."""

    @staticmethod
    def forward(ctx, y, mu, var, noise):
        S, n = mu.shape
        muc, varc, yc, nz = mu.detach().contiguous(), var.detach().contiguous(), y.detach().contiguous(), noise.detach()
        sums = torch.zeros(S, dtype=torch.float64, device=mu.device)
        sq = torch.zeros(S, dtype=torch.float64, device=mu.device)
        gmu, gvar = torch.empty_like(muc), torch.empty_like(muc)
        check(lib().npgp_gauss_ell_batched(S, n, ptr(yc), ptr(muc), ptr(varc), ptr(nz), 1.0, ptr(sums), ptr(sq),
                                           ptr(gmu), ptr(gvar), stream()), "npgp_gauss_ell_batched")
        ctx.save_for_backward(gmu, gvar, sq, nz)
        ctx.n = n
        return sums

    @staticmethod
    def backward(ctx, dsums):
        gmu, gvar, sq, nz = ctx.saved_tensors
        d = dsums.unsqueeze(-1)
        dnoise = (dsums * 0.5 * (sq / (nz * nz) - ctx.n / nz)).sum().reshape(nz.shape)
        return None, d * gmu, d * gvar, dnoise


def rbfper_fwd(t1, t2, hyp, out=None):
    """K = s * RBF(t1,t2) * Periodic(t1,t2) on 1-D inputs; hyp = [l_rbf, l_per, period, s] (4,).  `out` may be a strided
    view (e.g. the left half of a wider feature matrix)."""
    t1, t2, hyp = _c(t1.reshape(-1)), _c(t2.reshape(-1)), _c(hyp)
    K = out if out is not None else torch.empty(t1.numel(), t2.numel(), dtype=torch.float64, device=t1.device)
    check(lib().npgp_rbfper_fwd(t1.numel(), t2.numel(), ptr(t1), ptr(t2), ptr(hyp), ptr(K), K.stride(0), stream()),
          "npgp_rbfper_fwd")
    return K


def rbfper_bwd(t1, t2, hyp, G, need_dt2=False):
    """Gradients of sum(G * K) w.r.t. hyp (4,) and optionally t2.  G may be a strided view (row stride G.stride(0))."""
    t1, t2, hyp = _c(t1.reshape(-1)), _c(t2.reshape(-1)), _c(hyp)
    assert G.stride(1) == 1
    out4 = torch.zeros(4, dtype=torch.float64, device=G.device)
    dt2 = torch.zeros_like(t2) if need_dt2 else None
    check(lib().npgp_rbfper_bwd(t1.numel(), t2.numel(), ptr(t1), ptr(t2), ptr(hyp), ptr(G), G.stride(0), ptr(out4),
                                ptr(dt2), stream()), "npgp_rbfper_bwd")
    return out4, dt2


class RbfPerFn(torch.autograd.Function):
    """K = s * RBF(t1,t2) * Periodic(t1,t2) on 1-D inputs; hyp = [l_rbf, l_per, period, s] (4,).  Gradients to hyp, t2."""

    @staticmethod
    def forward(ctx, t1, t2, hyp):
        t1c, t2c, hc = t1.detach().contiguous().reshape(-1), t2.detach().contiguous().reshape(-1), hyp.detach().contiguous()
        K = rbfper_fwd(t1c, t2c, hc)
        ctx.save_for_backward(t1c, t2c, hc)
        ctx.t2_shape = t2.shape
        return K

    @staticmethod
    def backward(ctx, G):
        t1, t2, hyp = ctx.saved_tensors
        out4, dt2 = rbfper_bwd(t1, t2, hyp, G.contiguous(), need_dt2=ctx.needs_input_grad[1])
        return None, (dt2.reshape(ctx.t2_shape) if dt2 is not None else None), out4


def rbf_periodic(t1, t2, hyp):
    return RbfPerFn.apply(t1, t2, hyp)


def rowquad_sym(K, Cm):
    return RowquadFn.apply(K, Cm)


def dsvi_sample(mu, var, eps=None, seed=0, offset=0):
    return DsviSampleFn.apply(mu, var, eps, seed, offset)


def gauss_ell_batched(y, mu, var, noise):
    return GaussEllBatchedFn.apply(y, mu, var, noise)


def gibbs_diag(x1, ell1, x2, ell2, scale=None):
    return GibbsDiagFn.apply(x1, ell1, x2, ell2, scale)


def gibbs_full(x1, S1p, x2, S2p, scale=None, jitter=1e-5):
    return GibbsFullFn.apply(x1, S1p, x2, S2p, scale, jitter)


def sigma_from_h(H, Dm):
    return SigmaFromHFn.apply(H, Dm)


def rbf_matvec(x, z, lam, os, V, bias=None, apply_exp=False):
    return RbfMatvecFn.apply(x, z, lam, os, V, bias, apply_exp)


def status_update(status, info=None, loss=None):
    """Sticky device status: |= 1 if *info != 0, |= 2 if *loss is not finite."""
    check(lib().npgp_status_update(ptr(status), ptr(info), ptr(loss), stream()), "npgp_status_update")


def adam_step_guarded_(p, g, m, v, step_dev, status, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8, gscale=1.0, mask=None):
    """adam_step_dev_ that does nothing while *status != 0 (failed factorisation / non-finite loss in this or an earlier step)."""
    check(lib().npgp_adam_step_guarded(p.numel(), ptr(p), ptr(g), ptr(m), ptr(v), ptr(mask), float(lr), float(beta1),
                                       float(beta2), float(eps), ptr(step_dev), float(gscale), ptr(status), stream()),
          "npgp_adam_step_guarded")
    return p


def timestamp(buf, slot):
    """buf[slot] (int64, device) = GPU nanosecond timer at this point of the current stream (graph-capturable)."""
    check(lib().npgp_timestamp(ptr(buf), int(slot), stream()), "npgp_timestamp")


def available() -> bool:
    import os
    return os.path.exists(_lib.LIB_PATH)
