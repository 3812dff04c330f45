"""ctypes binding of libmpvae_b200.so (C-ABI declared in include/mpvae_b200.h).

No pybind, no torch types across the boundary: raw device pointers, sizes and the CUDA stream handle.
There is deliberately no fallback: if the shared library is missing (or a symbol is), importing this
module raises -- the product path must never silently run on anything but the CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmpvae_b200.so")

ABI_VERSION = 13
FLAG_SANITIZE_DEGENERATE = 0x1
FLAG_CONTRACT_TENSOR = 0x2
FLAG_CONTRACT_FMA = 0x4
FLAG_STABLE_CDF = 0x8
FLAG_FUSED_FORWARD = 0x10
FLAG_SEPARATE_NOISE = 0x20
FLAG_FUSED_EXCHANGE = 0x40
FLAG_SERIAL_EXCHANGE = 0x80
PEER_TILE_BYTES = 65536

# every symbol include/mpvae_b200.h declares
EXPORTS = (
    "mpvae_workspace_bytes", "mpvae_probit_forward", "mpvae_probit_predict", "mpvae_probit_backward", "mpvae_philox_normal",
    "mpvae_contract_nt", "mpvae_contract_nt_pitched", "mpvae_contract_tn", "mpvae_grad_norm_workspace",
    "mpvae_grad_norm", "mpvae_adam_step", "mpvae_tc_planes_bytes", "mpvae_tc_tail_scratch_bytes", "mpvae_tc_split",
    "mpvae_tc_gemm_nt", "mpvae_tc_gemm_tn", "mpvae_peer_flag_bytes", "mpvae_peer_allreduce", "mpvae_peer_allreduce_dev", "mpvae_peer_allreduce_nvls", "mpvae_label_curves",
    "mpvae_peer_alloc", "mpvae_peer_open", "mpvae_peer_close", "mpvae_peer_free", "mpvae_contract_workspace_bytes", "mpvae_last_error",
    "mpvae_abi_version", "mpvae_launch_count", "mpvae_batch_metrics", "mpvae_batch_metrics_workspace",
    "mpvae_peer_error", "mpvae_profile", "mpvae_profile_read", "mpvae_profile_name", "mpvae_test_log_normal",
    "mpvae_predictive_scale", "mpvae_predictive_rho", "mpvae_predict_exact", "mpvae_predict_pairs",
    "mpvae_probit_predict_conditional", "mpvae_probit_forward_masked", "mpvae_probit_backward_masked",
    "mpvae_ghk_workspace_bytes", "mpvae_probit_predict_conditional_ghk",
    "mpvae_probit_sample_labels", "mpvae_f1_sets_workspace_bytes", "mpvae_f1_sets",
)

_f = C.c_void_p  # device pointer


class ProbitParams(C.Structure):
    """Mirror of `mpvae_probit_params` (field order and types must match the header)."""
    _fields_ = [
        ("struct_bytes", C.c_uint32), ("flags", C.c_uint32),
        ("S", C.c_int32), ("B", C.c_int32), ("L", C.c_int32), ("Z", C.c_int32), ("D", C.c_int32),
        ("nll_coeff", C.c_float), ("c_coeff", C.c_float),
        ("y", _f), ("fe_out", _f), ("fx_out", _f), ("fe_mu", _f), ("fe_logvar", _f), ("fx_mu", _f),
        ("fx_logvar", _f), ("r", _f), ("noise", _f),
        ("scalars", _f * 6), ("indiv_prob", _f), ("indiv_prob_label", _f),
        ("g_scalars", _f * 6), ("g_indiv_prob", _f), ("g_indiv_prob_label", _f),
        ("g_fe_out", _f), ("g_fx_out", _f), ("g_fe_mu", _f), ("g_fe_logvar", _f), ("g_fx_mu", _f),
        ("g_fx_logvar", _f), ("g_r", _f),
        ("workspace", _f), ("workspace_bytes", C.c_uint64),
        ("noise_seed", C.c_uint64), ("noise_offset", C.c_uint64),
        ("noise_b_global", C.c_int32), ("noise_row0", C.c_int32),
        ("noise_offset_dev", _f),
        ("peer_world", C.c_int32), ("peer_rank", C.c_int32), ("peer_step", C.c_uint32), ("peer_reserved", C.c_uint32),
        ("peer_part", _f * 8), ("peer_g_r", _f * 8), ("peer_flags", _f * 8),
        ("peer_mc_part", _f), ("peer_mc_g_r", _f),
        ("peer_step_dev", _f),
        ("peer_tile_done", _f * 8),
    ]


# size of the struct up to (not including) peer_world: MPVAE_PARAMS_BASE_BYTES of the header
PARAMS_BASE_BYTES = ProbitParams.peer_world.offset


class LibraryMissing(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). mpvae_b200 has no CPU / eager fallback.")
    lib = C.CDLL(LIB_PATH)
    missing = [s for s in EXPORTS if not hasattr(lib, s)]
    if missing:
        raise LibraryMissing(f"{LIB_PATH} lacks symbols {missing}; rebuild")
    lib.mpvae_abi_version.restype = C.c_int
    if lib.mpvae_abi_version() != ABI_VERSION:
        raise LibraryMissing(f"ABI mismatch: library {lib.mpvae_abi_version()} vs binding {ABI_VERSION}; rebuild")
    lib.mpvae_last_error.restype = C.c_char_p
    lib.mpvae_launch_count.restype = C.c_uint64
    lib.mpvae_workspace_bytes.restype = C.c_uint64
    lib.mpvae_workspace_bytes.argtypes = [C.c_int32] * 5 + [C.c_uint32]
    lib.mpvae_probit_forward.restype = C.c_int
    lib.mpvae_probit_forward.argtypes = [C.POINTER(ProbitParams), C.c_void_p]
    lib.mpvae_probit_predict.restype = C.c_int
    lib.mpvae_probit_predict.argtypes = [C.POINTER(ProbitParams), C.c_void_p]
    lib.mpvae_probit_predict_conditional.restype = C.c_int
    lib.mpvae_probit_predict_conditional.argtypes = [C.POINTER(ProbitParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mpvae_ghk_workspace_bytes.restype = C.c_uint64
    lib.mpvae_ghk_workspace_bytes.argtypes = [C.c_int32] * 5 + [C.c_uint32]
    lib.mpvae_probit_predict_conditional_ghk.restype = C.c_int
    lib.mpvae_probit_predict_conditional_ghk.argtypes = [C.POINTER(ProbitParams)] + [C.c_void_p] * 5 + [
        C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mpvae_probit_sample_labels.restype = C.c_int
    lib.mpvae_probit_sample_labels.argtypes = [C.POINTER(ProbitParams), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mpvae_f1_sets_workspace_bytes.restype = C.c_uint64
    lib.mpvae_f1_sets_workspace_bytes.argtypes = [C.c_int32] * 3
    lib.mpvae_f1_sets.restype = C.c_int
    lib.mpvae_f1_sets.argtypes = [C.c_void_p] + [C.c_int32] * 3 + [C.c_double, C.c_int32] + [C.c_void_p] * 4 + [
        C.c_uint64, C.c_void_p]
    lib.mpvae_probit_backward.restype = C.c_int
    lib.mpvae_probit_backward.argtypes = [C.POINTER(ProbitParams), C.c_void_p]
    for fn in (lib.mpvae_probit_forward_masked, lib.mpvae_probit_backward_masked):
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(ProbitParams), C.c_void_p, C.c_void_p]
    lib.mpvae_philox_normal.restype = C.c_int
    lib.mpvae_philox_normal.argtypes = [C.c_void_p] + [C.c_int32] * 5 + [C.c_uint64, C.c_uint64, C.c_void_p]
    lib.mpvae_contract_workspace_bytes.restype = C.c_uint64
    lib.mpvae_contract_workspace_bytes.argtypes = [C.c_int32] * 4
    lib.mpvae_batch_metrics_workspace.restype = C.c_uint64
    lib.mpvae_batch_metrics_workspace.argtypes = [C.c_int32, C.c_int32]
    lib.mpvae_batch_metrics.restype = C.c_int
    lib.mpvae_batch_metrics.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                        C.c_uint64, C.c_void_p]
    lib.mpvae_predictive_scale.restype = C.c_int
    lib.mpvae_predictive_scale.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.mpvae_predictive_rho.restype = C.c_int
    lib.mpvae_predictive_rho.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                         C.c_void_p]
    lib.mpvae_predict_exact.restype = C.c_int
    lib.mpvae_predict_exact.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.mpvae_predict_pairs.restype = C.c_int
    lib.mpvae_predict_pairs.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                        C.c_uint32, C.c_void_p, C.c_void_p]
    for fn in (lib.mpvae_contract_nt, lib.mpvae_contract_tn):
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 4 + [C.c_void_p, C.c_uint64, C.c_void_p]
    lib.mpvae_label_curves.restype = C.c_int
    lib.mpvae_label_curves.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_void_p]
    lib.mpvae_peer_allreduce_nvls.restype = C.c_int
    lib.mpvae_peer_allreduce_nvls.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                              C.c_uint32, C.c_uint64, C.c_void_p]
    lib.mpvae_peer_allreduce_dev.restype = C.c_int
    lib.mpvae_peer_allreduce_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p,
                                             C.c_uint64, C.c_void_p]
    lib.mpvae_peer_allreduce.restype = C.c_int
    lib.mpvae_peer_allreduce.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint32, C.c_uint64,
                                         C.c_void_p]
    lib.mpvae_peer_flag_bytes.restype = C.c_uint64
    lib.mpvae_peer_flag_bytes.argtypes = []
    lib.mpvae_peer_alloc.restype = C.c_int
    lib.mpvae_peer_alloc.argtypes = [C.c_uint64, C.POINTER(C.c_void_p), C.c_char_p]
    lib.mpvae_peer_open.restype = C.c_int
    lib.mpvae_peer_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    lib.mpvae_peer_close.restype = C.c_int
    lib.mpvae_peer_close.argtypes = [C.c_void_p]
    lib.mpvae_peer_free.restype = C.c_int
    lib.mpvae_peer_free.argtypes = [C.c_void_p]
    lib.mpvae_tc_planes_bytes.restype = C.c_uint64
    lib.mpvae_tc_planes_bytes.argtypes = [C.c_int32, C.c_int32]
    lib.mpvae_tc_tail_scratch_bytes.restype = C.c_uint64
    lib.mpvae_tc_tail_scratch_bytes.argtypes = []
    lib.mpvae_tc_split.restype = C.c_int
    lib.mpvae_tc_split.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mpvae_tc_gemm_nt.restype = C.c_int
    lib.mpvae_tc_gemm_nt.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 4 + [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                                                         C.c_uint64, C.c_void_p]
    lib.mpvae_tc_gemm_tn.restype = C.c_int
    lib.mpvae_tc_gemm_tn.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 3 + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                                                         C.c_void_p]
    lib.mpvae_grad_norm_workspace.restype = C.c_uint64
    lib.mpvae_grad_norm_workspace.argtypes = []
    lib.mpvae_grad_norm.restype = C.c_int
    lib.mpvae_grad_norm.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_void_p, C.c_double, C.c_double,
                                    C.c_double, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.mpvae_adam_step.restype = C.c_int
    lib.mpvae_adam_step.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                    C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p]
    lib.mpvae_contract_nt_pitched.restype = C.c_int
    lib.mpvae_contract_nt_pitched.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 5 + [C.c_void_p, C.c_uint64, C.c_void_p]
    lib.mpvae_peer_error.restype = C.c_int
    lib.mpvae_peer_error.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]
    lib.mpvae_test_log_normal.restype = C.c_int
    lib.mpvae_test_log_normal.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.mpvae_profile.restype = C.c_int
    lib.mpvae_profile.argtypes = [C.c_int32]
    lib.mpvae_profile_read.restype = C.c_int
    lib.mpvae_profile_read.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    lib.mpvae_profile_name.restype = C.c_char_p
    lib.mpvae_profile_name.argtypes = [C.c_int32]
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().mpvae_last_error()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def launch_count() -> int:
    return int(lib().mpvae_launch_count())


def profile(enable: bool):
    """Switch the library's per-kernel CUDA-event timing on (and clear it) or off (include/mpvae_b200.h)."""
    check(lib().mpvae_profile(1 if enable else 0), "mpvae_profile")


def profile_read() -> dict:
    """{slot name: (total ms, launches recorded)} since the last `profile(True)`; waits for the recorded events."""
    out = {}
    slot = 0
    while True:
        name = lib().mpvae_profile_name(slot)
        if name is None:
            return out
        ms, n = C.c_double(), C.c_int32()
        check(lib().mpvae_profile_read(slot, C.byref(ms), C.byref(n)), "mpvae_profile_read")
        if n.value:
            out[name.decode()] = (ms.value, n.value)
        slot += 1
