"""ctypes binding of libnpgp.so (C ABI declared in include/npgp.h).

There is NO fallback: if the shared library is missing or a call fails, this raises.  PyTorch is used only to own device
memory and to name the CUDA stream the kernels are enqueued on."""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnpgp.so")

_p = C.c_void_p
_i = C.c_int
_l = C.c_long
_d = C.c_double



class SvgpConfig(C.Structure):
    """npgp_svgp_config of include/npgp.h (field for field)."""
    _fields_ = [("variant", C.c_int), ("d", C.c_int), ("M", C.c_int), ("B_local", C.c_int), ("N_total", C.c_long),
                ("B_global", C.c_int), ("world_size", C.c_int), ("jitter_zz", C.c_double), ("jitter_xx", C.c_double),
                ("kernel_jitter", C.c_double), ("min_var", C.c_double), ("extra_jitter", C.c_double), ("learn_z", C.c_int),
                ("include_prior", C.c_int), ("row_os", C.c_void_p), ("row_lam", C.c_void_p), ("prior_c", C.c_void_p),
                ("prior_os", C.c_void_p), ("prior_lam", C.c_void_p), ("timeline", C.c_void_p)]


_SIGS = {
    "npgp_version": ([], _i),
    "npgp_launch_count": ([], _l),
    "npgp_timestamp": ([_p, _i, _p], _i),
    "npgp_gibbs_diag_fwd": ([_i, _i, _i, _p, _p, _p, _p, _p, _p, _l, _p, _p, _p], _i),
    "npgp_gibbs_diag_bwd": ([_i, _i, _i, _p, _p, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p], _i),
    "npgp_gibbs_full_fwd": ([_i, _i, _i, _p, _p, _p, _p, _d, _p, _p, _l, _p, _p, _p], _i),
    "npgp_gibbs_full_bwd": ([_i, _i, _i, _p, _p, _p, _p, _d, _p, _p, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p], _i),
    "npgp_sigma_from_h_fwd": ([_i, _i, _p, _p, _p, _p], _i),
    "npgp_sigma_from_h_bwd": ([_i, _i, _p, _p, _p, _p, _p, _p], _i),
    "npgp_rbf_matvec_fwd": ([_i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _i, _p, _p], _i),
    "npgp_rbf_matvec_bwd": ([_i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p], _i),
    "npgp_dgemm": ([_i, _i, _i, _i, _i, _d, _p, _l, _p, _l, _d, _p, _l, _i, _i, _i, _p], _i),
    "npgp_rowquad": ([_i, _i, _p, _l, _p, _l, _p, _l, _p, _p], _i),
    "npgp_rowquad_i8_workspace_bytes": ([_i, _i], _l),
    "npgp_rowquad_i8_debug": ([_p], None),
    "npgp_rowquad_i8_slice_only": ([_i, _i, _p, _l, _p, _l, _p, _l, _p], _i),
    "npgp_rowquad_i8_gemm_only": ([_i, _i, _p, _l, _p, _l, _p, _p, _l, _p], _i),
    "npgp_syrk_i8_workspace_bytes": ([_i, _i], _l),
    "npgp_syrk_i8": ([_i, _i, _d, _p, _l, _p, _p, _d, _i, _i, _p, _l, _p, _l, _p], _i),
    "npgp_syrk_i8_prepare": ([_i, _i, _p, _l, _p, _p, _p, _l, _p], _i),
    "npgp_wsyrk_weighted_only": ([_i, _i, _d, _p, _l, _p, _p, _d, _p, _l, _p], _i),
    "npgp_rowquad_i8": ([_i, _i, _p, _l, _p, _l, _p, _l, _p, _p, _l, _p], _i),
    "npgp_o8_set_collector": ([_i], _i),
    "npgp_o8_set_syrk_split": ([_i], _i),
    "npgp_o8_digits_bytes": ([_i, _i, _i], _l),
    "npgp_o8_slice_rows": ([_i, _i, _p, _l, _i, _p, _p, _p], _i),
    "npgp_o8_rowquad_digits": ([_i, _i, _p, _p, _p, _p, _p, _p, _l, _p, _l, _p, _l, _p, _p, _p], _i),
    "npgp_o8_sum_partials": ([_i, _i, _p, _p, _p], _i),
    "npgp_o8_trinorm_digits": ([_i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _l, _p], _i),
    "npgp_o8_gemm_digits": ([_i, _i, _i, _p, _p, _p, _p, _p, _p, _l, _p], _i),
    "npgp_o8_syrk_part_bytes": ([_i, _i], _l),
    "npgp_o8_syrk_digits": ([_i, _i, _p, _p, _d, _p, _p, _p, _i, _p, _l, _p, _l, _p], _i),
    "npgp_gibbs_digits_splits": ([_i, _i], _i),
    "npgp_gibbs_full_fwd_digits": ([_i, _i, _i, _p, _p, _p, _p, _d, _p, _p, _p, _p, _l, _p], _i),
    "npgp_gibbs_diag_fwd_digits": ([_i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p], _i),
    "npgp_mu_gmu_parts": ([_i, _p, _p, _i, _l, _p, _d, _p, _p, _p], _i),
    "npgp_gauss_ell_parts_workspace_bytes": ([_i], _l),
    "npgp_gauss_ell_parts": ([_i, _p, _p, _p, _i, _l, _p, _d, _d, _p, _d, _p, _p, _p, _p, _p, _p, _p, _l, _p], _i),
    "npgp_wsyrk": ([_i, _i, _d, _p, _l, _p, _p, _l, _p], _i),
    "npgp_wsyrk_hint": ([_i, _i, _d, _p, _l, _p, _p, _d, _p, _l, _p], _i),
    "npgp_symmetrize": ([_i, _p, _l, _i, _p], _i),
    "npgp_trsm": ([_i, _i, _i, _p, _l, _p, _l, _p, _l, _p], _i),
    "npgp_potrf_workspace_bytes": ([_i], _l),
    "npgp_potrf_inv_lower": ([_i, _p, _l, _p, _l, _p, _l, _p, _p], _i),
    "npgp_potrf_flow_workspace_bytes": ([_i], _l),
    "npgp_potrf_inv_flow": ([_i, _p, _l, _p, _l, _p, _l, _p, _p], _i),
    "npgp_potrf_inv_flow_batch": ([_i, _i, _p, _l, _p, _l, _p, _l, _p, _p], _i),
    "npgp_fp64_peak_probe": ([_i, _i, _i, _p, _p], _i),
    "npgp_i8_peak_probe": ([_i, _i, _i, _i, _p], _i),
    "npgp_i8_peak_probe_pair": ([_i, _i, _i, _i, _p], _i),
    "npgp_set_gemm_config": ([_i], _i),
    "npgp_colwsum": ([_i, _i, _p, _l, _p, _p, _p], _i),
    "npgp_gemv_n": ([_i, _i, _p, _l, _p, _p, _p], _i),
    "npgp_gauss_ell": ([_i, _p, _p, _p, _p, _d, _d, _p, _d, _p, _p, _p, _p, _p], _i),
    "npgp_phi_mask": ([_i, _p, _l, _d, _p], _i),
    "npgp_adam_step": ([_l, _p, _p, _p, _p, _p, _d, _d, _d, _d, _i, _d, _p], _i),
    "npgp_adam_step_dev": ([_l, _p, _p, _p, _p, _p, _d, _d, _d, _d, _p, _d, _p], _i),
    "npgp_status_update": ([_p, _p, _p, _p], _i),
    "npgp_adam_step_guarded": ([_l, _p, _p, _p, _p, _p, _d, _d, _d, _d, _p, _d, _p, _p], _i),
    "npgp_rbfper_fwd": ([_i, _i, _p, _p, _p, _p, _l, _p], _i),
    "npgp_rbfper_bwd": ([_i, _i, _p, _p, _p, _p, _l, _p, _p, _p], _i),
    "npgp_dsvi_sample": ([_l, _p, _p, _p, C.c_ulonglong, C.c_ulonglong, _p, _p, _p], _i),
    "npgp_dsvi_sample_bwd": ([_l, _p, _p, _p, _p, _p, _p], _i),
    "npgp_gauss_ell_batched": ([_i, _i, _p, _p, _p, _p, _d, _p, _p, _p, _p, _p], _i),
    "npgp_dsvi_layer_workspace_bytes": ([_i, _i, _i], _l),
    "npgp_dsvi_layer_fwd": ([_i, _i, _i, _p, _p, _p, _p, _p, _p, _d, _d, _d, _p, _p, _p, _p, _l, _p], _i),
    "npgp_dsvi_layer_bwd": ([_i, _i, _i, _p, _p, _p, _p, _p, _p, _d, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p], _i),
    "npgp_svgp_theta_size": ([_p], _l),
    "npgp_svgp_workspace_bytes": ([_p], _l),
    "npgp_svgp_plan_create": ([_p, _p, _p, _l], _i),
    "npgp_svgp_plan_destroy": ([_p], _i),
    "npgp_svgp_set_extra_jitter": ([_p, _d], _i),
    "npgp_svgp_num_sections": ([], _i),
    "npgp_svgp_section_name": ([_i], C.c_char_p),
    "npgp_svgp_elbo_fwd": ([_p, _p, _p, _p, _p, _p, _p], _i),
    "npgp_svgp_elbo_bwd": ([_p, _p, _p, _p, _p], _i),
    "npgp_svgp_step": ([_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _d, _d, _d, _d, _p, _p], _i),
    "npgp_svgp_predict_prepare": ([_p, _p, _p, _p], _i),
    "npgp_svgp_predict": ([_p, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p], _i),
    "npgp_svgp_sample_workspace_bytes": ([_p, _i], _l),
    "npgp_svgp_sample_prepare": ([_p, _p, _i, C.c_ulonglong, _p, _l, _p], _i),
    "npgp_svgp_sample": ([_p, _l, _p, _l, _p, _i, _p, _l, _p, _l, _p], _i),
    "npgp_sample_normals": ([_i, _i, _i, C.c_ulonglong, _p, _p], _i),
    "npgp_svgp_buffer": ([_p, _i], _p),
    "npgp_sgpr_predict_workspace_bytes": ([_i], _l),
    "npgp_sgpr_predict_finish": ([_i, _p, _l, _i, _i, _p, _l, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p], _i),
    "npgp_sgpr_rownorm_parts": ([_i, _i, _p, _l, _p, _l, _p], _i),
    "npgp_sgpr_sample_finish": ([_i, _i, _p, _p, _l, _i, _i, _p, _l, _p, _p, _p, _i, C.c_ulonglong, _l, _p, _l, _p], _i),
    "npgp_comm_unique_id": ([_p], _i),
    "npgp_comm_create": ([_p, _p, _i, _i], _i),
    "npgp_comm_destroy": ([_p], _i),
    "npgp_allreduce_f64": ([_p, _p, _l, _p], _i),
    "npgp_allreduce_f64_pair": ([_p, _p, _l, _p, _l, _p], _i),
}

_lib = None


class NpgpError(RuntimeError):
    pass


def exported_symbols():
    return sorted(_SIGS)


def lib():
    """Load libnpgp.so (once).  Raises if it has not been built -- there is no CPU or eager fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NpgpError(
                "libnpgp.so not found at %s: build it with `python -m nonstationary_precip_b200.build` "
                "(the CUDA extension is mandatory; there is no fallback path)" % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in _SIGS.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = restype
        if os.environ.get("NPGP_O8_COLLECTOR") == "0":  # measurement / debugging switch (see npgp_o8_set_collector)
            handle.npgp_o8_set_collector(0)
        _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc == 0:
        return
    if rc < 0:
        msg = {-1: "invalid argument", -2: "unsupported configuration", -3: "workspace too small"}.get(rc, "error")
    else:
        msg = "CUDA error %d" % rc
    raise NpgpError("%s failed: %s" % (what, msg))


def ptr(t):
    """Raw device pointer of a CUDA fp64 tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NpgpError("npgp kernels need CUDA tensors (got a %s tensor); there is no CPU path" % t.device.type)
    if t.dtype not in (torch.float64, torch.int32, torch.uint8, torch.int8, torch.int64):
        raise NpgpError("npgp kernels take fp64 data (int32 exponents / indices, uint8 digit planes); got %s" % t.dtype)
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream
