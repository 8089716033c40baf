"""ctypes binding of libpxmcmc_b200.so (the C ABI in include/pxmcmc_b200.h)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PXM_LIB", os.path.join(_HERE, "libpxmcmc_b200.so"))

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m pxmcmc_b200.build` "
        "(nvcc, sm_100a).  pxmcmc_b200 has no CPU fallback."
    )

lib = C.CDLL(LIB_PATH)

_vp, _i, _ll, _d, _u64, _u32 = C.c_void_p, C.c_int, C.c_longlong, C.c_double, C.c_ulonglong, C.c_uint

# every symbol include/pxmcmc_b200.h declares, with its argument types
SIGNATURES = {
    "pxm_last_error": (C.c_char_p, []),
    "pxm_init": (_i, [_i]),
    "pxm_sht_plan_create": (_i, [_i, _i, _i, C.POINTER(_vp)]),
    "pxm_sht_plan_destroy": (_i, [_vp]),
    "pxm_sht_plan_table_bytes": (C.c_size_t, [_vp]),
    "pxm_sht_inverse": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "pxm_sht_forward": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "pxm_sht_inverse_adjoint": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "pxm_sht_forward_adjoint": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "pxm_wav_plan_create": (_i, [_i, _d, _i, _i, C.POINTER(_vp)]),
    "pxm_wav_plan_destroy": (_i, [_vp]),
    "pxm_wav_plan_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_ll), C.POINTER(_ll), C.POINTER(_i), C.POINTER(_ll)]),
    "pxm_wav_plan_bandlimits": (_i, [_vp, C.POINTER(_i), _i]),
    "pxm_wav_plan_table_bytes_by_family": (_i, [_vp, C.POINTER(_ll)]),
    "pxm_wav_plan_gram_bytes": (_i, [_vp, C.POINTER(_ll)]),
    "pxm_wav_set_gram_weights": (_i, [_vp, C.POINTER(C.c_double), _i]),
    "pxm_wav_synthesis": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_synthesis_adjoint": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_analysis": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_analysis_adjoint": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_synthesis_harmonic": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_synthesis_adjoint_harmonic": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_ring_doubles": (_ll, [_vp]),
    "pxm_wav_synthesis_to_ring": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_synthesis_adjoint_from_ring": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_ring_to_pix": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_pix_to_ring": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_ring_resid": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "pxm_wav_harm_doubles": (_ll, [_vp]),
    "pxm_wav_synthesis_to_harm": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_gram_gradient": (_i, [_vp, _vp, _vp, _d, _d, _vp, _i, _vp]),
    "pxm_wav_harm_to_pix": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wav_pix_to_harm_adjoint": (_i, [_vp, _vp, _vp, _i, _vp]),
    "pxm_wavelet_tiling": (_i, [_i, _d, _i, _vp, _vp, C.POINTER(_i)]),
    "pxm_hpx_plan_create": (_i, [_i, _i, C.POINTER(_vp)]),
    "pxm_hpx_plan_destroy": (_i, [_vp]),
    "pxm_hpx_alm2map": (_i, [_vp, _vp, _vp, _vp]),
    "pxm_hpx_map2alm_adjoint": (_i, [_vp, _vp, _vp, _vp]),
    "pxm_sht_plan_create_sharded": (_i, [_i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "pxm_wav_plan_create_sharded": (_i, [_i, _d, _i, _i, _i, _i, C.POINTER(_vp)]),
    "pxm_sht_plan_prepare": (_i, [_vp]),
    "pxm_wav_plan_prepare": (_i, [_vp]),
    "pxm_sht_plan_workspace": (_vp, [_vp, C.POINTER(C.c_size_t)]),
    "pxm_wav_plan_workspace": (_vp, [_vp, C.POINTER(C.c_size_t)]),
    "pxm_sht_plan_attach": (_i, [_vp, C.POINTER(_vp)]),
    "pxm_wav_plan_attach": (_i, [_vp, C.POINTER(_vp)]),
    "pxm_sht_plan_local_rows": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "pxm_wav_plan_local_rows": (_i, [_vp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_ll), C.POINTER(_ll)]),
    "pxm_sht_plan_barrier_status": (_i, [_vp, C.POINTER(_ll)]),
    "pxm_wav_plan_barrier_status": (_i, [_vp, C.POINTER(_ll)]),
    "pxm_shard_owner_of_m": (_i, [_i, _i]),
    "pxm_shard_ring_range": (_i, [_i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "pxm_ipc_export": (_i, [_vp, _vp]),
    "pxm_ipc_open": (_i, [_vp, C.POINTER(_vp)]),
    "pxm_ipc_close": (_i, [_vp]),
    "pxm_soft": (_i, [_i, _vp, _vp, _d, _vp, _ll, _ll, _vp]),
    "pxm_myula_update": (_i, [_vp, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp, _ll, _ll, _d, _d, _i, _u64, _u64, _u32, _vp]),
    "pxm_myula_update_dstep": (_i, [_vp, _vp, _vp, _vp, _d, _vp, _vp, _ll, _ll, _d, _d, _i, _u64, _vp, _u32, _vp]),
    "pxm_counter_add": (_i, [_vp, _u64, _vp]),
    "pxm_philox_normal": (_i, [_vp, _ll, _ll, _u64, _u64, _vp, _u32, _vp]),
    "pxm_myula_update_dpar": (_i, [_vp, _vp, _vp, _vp, _d, _vp, _vp, _ll, _ll, _vp, _i, _u64, _u64, _u32, _vp]),
    "pxm_reduce_dpar": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _d, _ll, _ll, _vp, _vp, _vp]),
    "pxm_pxmala_accept": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _ll, _u64, _u64, _u32, _vp, _vp, _ll, _i, _vp]),
    "pxm_select_if": (_i, [_vp, _ll, _ll, _vp, _vp, _vp, _i, _vp]),
    "pxm_resid_invcov": (_i, [_vp, _vp, _vp, _vp, _ll, _ll, _vp]),
    "pxm_reduce_scratch_elems": (_i, []),
    "pxm_reduce": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _d, _d, _ll, _ll, _vp, _vp, _vp]),
    "pxm_lincomb": (_i, [_i, C.POINTER(_vp), C.POINTER(_d), _vp, _d, _d, _vp, _ll, _vp]),
    "pxm_gradlogpi": (_i, [_vp, _vp, _vp, _d, _vp, _d, _vp, _ll, _ll, _vp]),
    "pxm_skrock_shift": (_i, [_vp, _d, _vp, _vp, _i, _u64, _u64, _vp, _u32, _vp, _ll, _ll, _vp]),
    "pxm_skrock_stage": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _d, _d, _d, _d, _d, _d, _vp, _vp, _i, _u64, _u64, _vp,
                              _u32, _vp, _ll, _ll, _vp]),
    "pxm_fista_update": (_i, [_vp, _vp, _vp, _vp, _d, _d, _d, _vp, _vp, _vp, _vp, _ll, _ll, _ll, _vp, _vp]),
    "pxm_masked_gather":(_i, [_vp, _vp, _vp, _vp, _ll, _ll, _ll, _vp]),
    "pxm_masked_scatter": (_i, [_vp, _vp, _vp, _vp, _ll, _ll, _ll, _vp]),
    "pxm_real_to_complex": (_i, [_vp, _vp, _ll, _vp]),
    "pxm_csr_spmv": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _ll, _ll, _vp]),
    "pxm_gc_count_points": (_i, [_vp, _vp, _ll, _d, _vp, _vp]),
    "pxm_gc_rasterise": (_i, [_vp, _vp, _ll, _i, _d, _i, _vp, _vp, _vp, _vp]),
    "pxm_gc_compact": (_i, [_vp, _vp, _vp, _i, _ll, _vp, _vp, _vp]),
    "pxm_quantile_columns": (_i, [_vp, _ll, _ll, _ll, _ll, _d, _ll, _d, _vp, _vp, _vp]),
    "pxm_quantile_columns_max_samples": (_i, []),
    "pxm_stats_accumulator_doubles": (_ll, [_ll, _ll, _i]),
    "pxm_stats_reset": (_i, [_vp, _ll, _ll, _i, _vp]),
    "pxm_stats_accumulate": (_i, [_vp, _vp, _ll, _ll, _i, _ll, _ll, _vp, _vp]),
    "pxm_stats_partials": (_i, [_vp, _ll, _ll, _i, _ll, _vp, _vp, _vp, _vp]),
    "pxm_rank_diagnostics_scratch_doubles": (_ll, [_ll, _ll, _ll]),
    "pxm_rank_diagnostics": (_i, [_vp, _ll, _ll, _ll, _ll, _vp, _vp, _vp, _vp, _vp]),
    "pxm_credible_state_doubles": (_ll, [_ll, _i, _ll, _ll, _ll]),
    "pxm_credible_reset": (_i, [_vp, _ll, _i, _ll, _ll, _ll, _vp]),
    "pxm_credible_push": (_i, [_vp, _vp, _ll, _ll, _i, _ll, _ll, _ll, _ll, _vp, _vp]),
    "pxm_credible_finalize": (_i, [_vp, _ll, _i, _ll, _ll, _d, _ll, _d, _vp, _vp, _vp]),
    "pxm_profile_begin": (_i, [_i]),
    "pxm_profile_end": (_i, [C.POINTER(_d), C.POINTER(_ll)]),
    "pxm_launch_count": (_ll, []),
    "pxm_debug_set_naive": (_i, [_i]),
    "pxm_debug_set_fft_multipass": (_i, [_i]),
    "pxm_debug_wigner_row_host": (_i, [_i, _i, _i, _i, _i, _vp]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)  # AttributeError here == header/library mismatch
    _f.restype = _res
    _f.argtypes = _args


class PxmError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise PxmError(lib.pxm_last_error().decode())


_initialised = False


def ensure_device():
    """Select the CUDA device torch is using; raises if there is none (no CPU fallback)."""
    global _initialised
    if _initialised:
        return
    import torch

    if not torch.cuda.is_available():
        raise PxmError("pxmcmc_b200 needs a CUDA (sm_100a) device: there is no CPU fallback")
    check(lib.pxm_init(torch.cuda.current_device()))
    _initialised = True


def stream_ptr():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """device pointer of a torch tensor (or None)"""
    return None if t is None else C.c_void_p(t.data_ptr())


def wavelet_tiling_host(L, B, J_min):
    """(J_max, kappa0[L], kappa[nscales, L]) -- host only, no GPU needed."""
    J = C.c_int(0)
    jmax = int(np.ceil(np.log(L) / np.log(B)))
    k0 = np.zeros(L)
    k = np.zeros((max(jmax - J_min + 1, 1), L))
    check(lib.pxm_wavelet_tiling(L, float(B), J_min, k0.ctypes.data, k.ctypes.data, C.byref(J)))
    assert J.value == jmax
    return J.value, k0, k


def wigner_row_host(grid_L, ring, m, spin, lmax):
    out = np.zeros(lmax)
    check(lib.pxm_debug_wigner_row_host(grid_L, ring, m, spin, lmax, out.ctypes.data))
    return out
