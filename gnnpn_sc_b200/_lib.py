"""ctypes binding of ``libgnnpn_b200.so`` (the C ABI declared in ``include/gnnpn_b200.h``).

There is no CPU fallback: if the shared library is missing or cannot be loaded
every operator raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C gnnpn_sc_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgnnpn_b200.so")

_lock = threading.Lock()
_lib = None

_p = C.c_void_p
_i64 = C.c_int64
_i = C.c_int
_f = C.c_float

# name -> (restype, argtypes); must list every symbol of include/gnnpn_b200.h
SIGNATURES = {
    "gnnpn_abi_version": (_i, []),
    "gnnpn_error_string": (C.c_char_p, [_i]),
    "gnnpn_launch_count": (C.c_uint64, []),
    "gnnpn_pn_packed_lstm_floats": (C.c_size_t, [_i, _i]),
    "gnnpn_pn_pack_lstm_f32": (_i, [_p] * 7 + [_i, _i, _p, _p]),
    "gnnpn_set_option": (_i, [C.c_char_p, _i]),
    "gnnpn_get_option": (_i, [C.c_char_p, C.POINTER(_i)]),
    "gnnpn_pn_input_limit": (_f, []),
    "gnnpn_pn_check_inputs_f32": (_i, [_p, _i64, _p, _p]),
    "gnnpn_pn_enc_layout": (_i, [_i64, _i, _i, _i, _i, _i]),
    "gnnpn_pn_enc_out_floats": (C.c_size_t, [_i64, _i, _i, _i]),
    "gnnpn_pn_enc_to_rowmajor_f32": (_i, [_p, _i64, _i, _i, _p, _p]),
    "gnnpn_lstm_encode_f32": (_i, [_p, _i64, _i, _i, _i, _p, _p, _p, _p, C.c_size_t, _i, _p]),
    "gnnpn_pn_workspace_bytes": (C.c_size_t, [_i64, _i]),
    "gnnpn_pn_decode_greedy_f32": (_i, [_p, _p, _p, _p, _f, _p, _i, _p, _i, _f, _i64, _i, _i, _i, _i, _i,
                                        _p, _p, _p, _p, _p, _p, _p, C.c_size_t, _i, _p]),
    "gnnpn_pn_rollouts_workspace_bytes": (C.c_size_t, [_i64, _i, _i]),
    "gnnpn_pn_decode_rollouts_f32": (_i, [_p, _p, _p, _p, _f, _p, _i, _p, _i, _f, _i64, _i, _i, _i, _i, _i,
                                          _p, _p, _p, _p, _p, _p, C.c_size_t, _i, _i, _p]),
    "gnnpn_pn_best_rollout_f32": (_i, [_p, _p, _i64, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "gnnpn_pn_train_forward_workspace_bytes": (C.c_size_t, [_i64, _i, _i, _i, _i, _i]),
    "gnnpn_pn_train_forward_f32": (_i, [_p, _p, _p, _p, _p, _p, _f, _i, _f, _i64, _i, _i, _i, _i, _i] + [_p] * 10 +
                                   [C.c_size_t, _p]),
    "gnnpn_pn_train_backward_workspace_floats": (C.c_size_t, [_i64, _i, _i, _i]),
    "gnnpn_pn_train_backward_f32": (_i, [_p] * 12 + [_i, _f, _i64, _i, _i, _i, _i, _p, _p, _p, C.c_size_t, _p]),
    "gnnpn_pn_att_block_floats": (C.c_size_t, [_i]),
    "gnnpn_pn_decode_general_workspace_bytes": (C.c_size_t, [_i64, _i, _i, _i, _i, _i, _i]),
    "gnnpn_pn_decode_general_f32": (_i, [_p, _p, _p, _p, _f, _p, _i, _p, _i, _i, _f, _i64, _i, _i, _i, _i, _i,
                                         _p, _p, _p, _p, _p, _p, _p, _p, _i, _p, C.c_size_t, _p]),
    "gnnpn_pn_ref_transform_f32": (_i, [_p, _p, _i64, _i, _p, _p]),
    "gnnpn_pn_query_transform_f32": (_i, [_p, _i64, _p, _i64, _i, _p, _i64, _p]),
    "gnnpn_pn_full_logits_bahdanau_f32": (_i, [_p, _p, _p, _p, _i, _f, _i64, _i, _i, _i, _p, _p]),
    "gnnpn_pn_full_logits_f32": (_i, [_p, _p, _p, _i, _p, _i, _f, _i64, _i, _i, _i, _p, _p]),
    "gnnpn_pn_anyh_workspace_floats": (C.c_size_t, [_i64, _i, _i]),
    "gnnpn_lstm_encode_anyh_f32": (_i, [_p, _i64, _i, _i, _i, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "gnnpn_pn_decode_anyh_f32": (_i, [_p, _p, _p, _p, _f, _p, _p, _p, _i, _f, _i64, _i, _i, _i, _i, _i,
                                      _p, _p, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "gnnpn_pn_full_logits_anyh_f32": (_i, [_p, _p, _p, _i, _f, _i64, _i, _i, _i, _p, _p]),
    "gnnpn_pn_attention_windows_f32": (_i, [_p, _p, _p, _f, _i, _f, _i64, _i, _i, _i, _i, _p, _p, _p, _p]),
    "gnnpn_pn_reward_f32": (_i, [_p, _p, _i64, _i, _i, _i, _i, _p, _p, _p, _p]),
    "gnnpn_woa_fitness_f64": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i, _p, _p, _p, _p]),
    "gnnpn_ml2pn_score_f64": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i, _p, _p, _p, _p]),
    "gnnpn_woa_search_f64": (_i, [_p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _p]),
    "gnnpn_woa_prepare_f64": (_i, [_p, _p, _p, _i64, _i] + [_p] * 7 + [_i64, _i, C.c_double] + [_p] * 12),
    "gnnpn_woa_prepare_rows": (_i64, [_i64, _i64, _i]),
    "gnnpn_pn_greedy_low_high_host": (_i, [_p, _i64, _i, _i, _i, _i, _i, _p, _p, _i, _f, _f, _p, _p, _p]),
    "gnnpn_select_candidates_f32": (_i, [_p, _i64, _p, _p, _i, _p, _p, _p, _i64, _i, _i, _i, _p, _p, _p]),
    "gnnpn_csr_build_workspace_bytes": (_i, [_i64, _i64, _i, C.POINTER(C.c_size_t)]),
    "gnnpn_csr_build": (_i, [_p, _p, _i64, _i64, _i, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "gnnpn_embed_concat_f32": (_i, [_p, _i64, _i, _p, _i, _i, _p, _i64, _p]),
    "gnnpn_spmm_csr_workspace_bytes": (C.c_size_t, [_i64, _i, _i64]),
    "gnnpn_spmm_csr_f32": (_i, [_p, _p, _p, _p, _i64, _p, _i64, _i64, _i64, _i, _f, _i, _p, _p, _p, _i, _i64, _p,
                                C.c_size_t, _p]),
    "gnnpn_bn_train_forward_f32": (_i, [_p, _i64, _i64, _i, _p, _p, _f, _f, _i, _p, _i64, _p, _p, _p, _p, _p]),
    "gnnpn_bn_train_backward_f32": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i, _p, _p, _p, _i, _p, _i64, _p, _p, _p]),
    "gnnpn_gemm_workspace_bytes": (C.c_size_t, [_i64, _i, _i]),
    "gnnpn_gemm_f32_bias_act": (_i, [_p, _i64, _p, _i64, _p, _p, _p, _i, _p, _i64, _i64, _i, _i, _p, C.c_size_t, _p]),
}


class GnnpnError(RuntimeError):
    pass


def lib():
    """The loaded library (loaded once).  Raises ``GnnpnError`` when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise GnnpnError(
                    f"{LIB_PATH} is not built; the CUDA extension is required (no CPU fallback). "
                    "Run __graft_entry__.build() or `make -C gnnpn_sc_b200/csrc`.")
            h = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(h, name)          # AttributeError if the ABI lost a symbol
                fn.restype = res
                fn.argtypes = args
            if h.gnnpn_abi_version() != 12:
                raise GnnpnError("libgnnpn_b200.so ABI version mismatch")
            _lib = h
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().gnnpn_error_string(rc).decode()
        raise GnnpnError(f"{what or 'gnnpn call'} failed: {msg} (code {rc})")


def set_option(name: str, value: int) -> None:
    """``gnnpn_set_option``: "scan" (-1 auto / 0 CTA-pair / 1 column-split), "scan_groups", "persistent", "prof",
    "bptt" (0: per-step BPTT kernels)."""
    check(lib().gnnpn_set_option(name.encode(), int(value)), f"set_option({name})")


def get_option(name: str) -> int:
    v = _i(0)
    check(lib().gnnpn_get_option(name.encode(), C.byref(v)), f"get_option({name})")
    return int(v.value)


def launch_count() -> int:
    return int(lib().gnnpn_launch_count())
