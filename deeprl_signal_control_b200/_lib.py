"""Loader of the native library (csrc/libtsc.so, C ABI of include/tsc.h).

There is deliberately NO fallback: if the CUDA library is missing or does not load, importing
the simulator fails loudly (the product path never routes through a CPU implementation).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("TSC_LIB", os.path.join(CSRC, "libtsc.so"))   # TSC_LIB: tuning variants only
_lib = None

# every symbol include/tsc.h declares
SYMBOLS = ["tsc_last_error", "tsc_create", "tsc_destroy", "tsc_reset", "tsc_set_train_mode",
           "tsc_observe", "tsc_step", "tsc_step_host", "tsc_step_host_range", "tsc_step_host_range_async", "tsc_set_record", "tsc_step_record", "tsc_get_trips", "tsc_get_counts", "tsc_get_traffic_stats",
           "tsc_dump_state", "tsc_info", "tsc_mean_live",
           # include/tsc_learn.h
           "tscl_create", "tscl_destroy", "tscl_fc_embed", "tscl_lstm_seq_fwd", "tscl_heads", "tscl_returns",
           "tscl_heads_loss", "tscl_lstm_seq_bwd", "tscl_fc_bwd", "tscl_fc_bwd_tc", "tscl_wgrad_tc", "tscl_clip_rmsprop",
           "tscl_pack_weights", "tscl_policy_step", "tscl_policy_step_v2", "tscl_policy_step_v2r", "tscl_unpack_store", "tscl_pack_wht", "tscl_lstm_seq_bwd_tc", "tscl_pack_wxt", "tscl_lstm_seq_bwd_tc_dx", "tscl_dx_tc", "tscl_host_transition", "tscl_device_transition", "tscl_memcpy_async", "tscl_fc_hidden_fwd", "tscl_fc_hidden_bwd", "tscl_debug_policy_prof", "tscl_debug_bptt_prof",
           "tscl_iql_create", "tscl_iql_destroy", "tscl_iql_forward", "tscl_iql_sample", "tscl_iql_td_grad",
           "tscl_iql_clip_adam", "tscl_iql_transition"]


def build_native(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a with nvcc (cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC] + (["-B"] if force else [])
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("nvcc build of libtsc.so failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout + out.stderr)
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "native library %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        _lib.tsc_last_error.restype = C.c_char_p
        for s in SYMBOLS:
            getattr(_lib, s)  # AttributeError here = ABI drift
    return _lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError("libtsc: " + lib().tsc_last_error().decode())
