"""ctypes binding of libcoda_b200.so (the C ABI in include/coda_b200.h).

There is no CPU fallback: importing works anywhere (so the symbol table can be checked
without a GPU), but every compute entry point needs an sm_100 device and ``require_device``
fails loudly without one.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

from . import build as _build

_LIB = None

OK = 0
VERSION = 202
MAX_WORLD = 16
REC_WORDS = 8
FLAG_NONFINITE_INPUT = 0x01
FLAG_RANGE_INPUT = 0x02
FLAG_NONFINITE_TABLE = 0x04
FLAG_NONFINITE_PI = 0x08
FLAG_NONFINITE_PBEST = 0x10
FLAG_NONFINITE_EIG = 0x20
FLAG_NO_CANDIDATE = 0x40
FLAG_XCHG_TIMEOUT = 0x80
FLAG_NEGATIVE_PROB = 0x100
FLAG_ROWSUM_WARN = 0x200
FLAG_PIPELINE_TIMEOUT = 0x400
FLAG_NAMES = {
    FLAG_NONFINITE_INPUT: "preds", FLAG_RANGE_INPUT: "preds range", FLAG_NONFINITE_TABLE: "pdf/cdf/integrand",
    FLAG_NONFINITE_PI: "pi_hat_xi", FLAG_NONFINITE_PBEST: "Pbest", FLAG_NONFINITE_EIG: "Pbest(beta) normalized",
}

p, i32, i64, f64, f32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_float, C.c_size_t


class XchgStruct(C.Structure):
    """coda_xchg_t (include/coda_b200.h)."""
    _fields_ = [("world", i32), ("rank", i32), ("box", p * MAX_WORLD), ("epoch", p), ("H", i32), ("C", i32),
                ("rep_words", i32)]


class StepStruct(C.Structure):
    """coda_step_t (include/coda_b200.h): one shard's device state as the fused step kernels see it."""
    _fields_ = [
        ("H", i32), ("C", i32), ("N", i64), ("n_offset", i64), ("fx_shift", i32), ("lr", f32),
        ("hard", p), ("labeled", p), ("D", p), ("jvec", p), ("sel", p),
        ("terms", p), ("slot_of_model", p), ("shadow_off", i64), ("shadow_col_stride", i64), ("model_stride", i64),
        ("have_ens", i32), ("compact_k", i32),
        ("pisum_fx", p), ("PB", p), ("pi_hat", p), ("m0", p), ("h_before", p), ("best_model", p),
        ("partials", p), ("nblocks", i32), ("eig", p), ("bestrec", p),
        ("labels_global", p), ("hist_idx", p), ("hist_q", p), ("hist_tie", p), ("hist_cap", i64), ("step_ctr", p),
        ("flags", p),
    ]


PX, PS = C.POINTER(XchgStruct), C.POINTER(StepStruct)

# name -> (restype, argtypes); mirrors include/coda_b200.h one to one
SIGNATURES = {
    "coda_b200_last_error": (C.c_char_p, []),
    "coda_b200_version": (i32, []),
    "coda_b200_sm_count": (i32, []),
    "coda_b200_device_check": (i32, []),
    "coda_b200_set_l2_fetch_granularity": (i32, [i32]),
    "coda_b200_xchg_box_bytes": (sz, [i32, i32, i32, i32]),
    "coda_b200_xchg_alloc": (i32, [sz, C.POINTER(p)]),
    "coda_b200_xchg_free": (i32, [p]),
    "coda_b200_ipc_export": (i32, [p, p]),
    "coda_b200_ipc_open": (i32, [p, C.POINTER(p)]),
    "coda_b200_ipc_close": (i32, [p]),
    "coda_b200_peer_enable": (i32, [i32]),
    "coda_b200_scan_slab": (i32, [p, i64, i32, i64, i32, p, p, p, p, p, p]),
    "coda_b200_confusion_accum": (i32, [p, i64, p, i32, i64, i32, i32, p, p]),
    "coda_b200_confusion_sorted": (i32, [p, i64, p, p, i32, i64, i32, i32, p, p]),
    "coda_b200_init_dirichlets": (i32, [p, p, i32, i32, i32, f64, f64, i32, p, p]),
    "coda_b200_scan_compact": (i32, [p, p, i64, i32, i64, i32, i32, p, p, p, p, p, p]),
    "coda_b200_confusion_compact": (i32, [p, p, i64, p, i32, i64, i32, i32, i32, p, p, p]),
    "coda_b200_pi_full_compact": (i32, [p, p, i64, p, i32, i64, i32, i32, p, p, p, p]),
    "coda_b200_pi_rank1_compact": (i32, [p, p, i64, p, i32, i64, i32, i32, p, f64, i32, p, p, p, p, p]),
    "coda_b200_compact_index_count": (i32, [p, i64, i32, i64, i32, i32, p, p]),
    "coda_b200_compact_index_fill": (i32, [p, p, i64, i32, i64, i32, i32, p, p, p, p]),
    "coda_b200_pi_rank1_index": (i32, [p, p, p, p, i32, i64, i32, p, f64, i32, p, p, p, p, p, p]),
    "coda_b200_pi_full": (i32, [p, i64, p, i32, i64, i32, p, p]),
    "coda_b200_pi_full_tc_ok": (i32, [i32, i64, i32, i64]),
    "coda_b200_pi_full_tc_scratch_bytes": (sz, [i32, i32]),
    "coda_b200_pi_full_tc": (i32, [p, i64, p, i32, i64, i32, p, p, p, p]),
    "coda_b200_pi_reduce": (i32, [p, i64, i32, i32, p, p, p, p]),
    "coda_b200_shadow_build": (i32, [p, i64, i32, i64, i32, p, i32, i64, p, p]),
    "coda_b200_pi_rank1": (i32, [p, p, i32, i64, i32, p, f64, i32, p, p, p, p, i32, i32, p]),
    "coda_b200_scan_slab_f16": (i32, [p, i64, i32, i64, i32, p, p, p, p, p, p]),
    "coda_b200_confusion_accum_f16": (i32, [p, i64, p, i32, i64, i32, i32, p, p]),
    "coda_b200_confusion_sorted_f16": (i32, [p, i64, p, p, i32, i64, i32, i32, p, p]),
    "coda_b200_pi_full_f16": (i32, [p, i64, p, i32, i64, i32, p, p]),
    "coda_b200_pi_full_tc_ok_f16": (i32, [i32, i64, i32, i64]),
    "coda_b200_pi_full_tc_f16": (i32, [p, i64, p, i32, i64, i32, p, p, p, p]),
    "coda_b200_shadow_build_f16": (i32, [p, i64, i32, i64, i32, p, i32, i64, p, p]),
    "coda_b200_pi_rank1_f16": (i32, [p, p, i32, i64, i32, p, f64, i32, p, p, p, p, i32, i32, p]),
    "coda_b200_tables_scratch_bytes": (sz, [i32, i32]),
    "coda_b200_beta_tables": (i32, [p, p, i32, i32, i32, f64, i32, i32, p, p, p, p, p, p, p, p, p, p]),
    "coda_b200_pair_count": (i32, [p, i32, i64, i32, p, p, p, p]),
    "coda_b200_pair_fill": (i32, [p, i32, i64, i32, p, p, p, p, p, p, p, p, p, p]),
    "coda_b200_pair_rows": (i32, [p, i32, i32, p, p, p, p, p, p, p, p, i32, p, p, p, p, p, p]),
    "coda_b200_pair_rows_tc": (i32, [p, i32, i32, p, p, p, p, p, p, p, i32, p, p, p, p, p, p]),
    "coda_b200_template_gains": (i32, [p, i32, i32, p, p, p, p, p]),
    "coda_b200_eig_blocks": (i32, [i64, i32, i32]),
    "coda_b200_gain_eig": (i32, [p, i64, i32, i32, p, p, p, p, p, p, p, p, p, p, p, i64, i32, p, p, i32, p, p, p, p]),
    "coda_b200_ell_build": (i32, [p, p, p, i64, i32, p, p, p]),
    "coda_b200_row_gains": (i32, [p, p, i64, i32, i32, p, p, p, p, p]),
    "coda_b200_step_select": (i32, [PS, PX, p]),
    "coda_b200_step_merge": (i32, [PS, PX, p]),
    "coda_b200_step_label": (i32, [PS, PX, p]),
    "coda_b200_step_mixture": (i32, [PS, PX, p]),
    "coda_b200_ties": (i32, [p, i64, p, p, i64, p, i32, p, p, p, p]),
    "coda_b200_report_gather": (i32, [p, i32, p, PX, p, p]),
}


class NativeError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """dlopen the in-tree library (building it with nvcc first if it is not there)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if build_if_missing and not os.environ.get("CODA_B200_NO_BUILD"):
        try:
            _build.build()            # no-op when the in-tree .so matches the sources
        except Exception as e:        # e.g. no nvcc on this box: use the shipped .so ONLY if it was built from these sources
            if not os.path.exists(path):
                raise NativeError(f"cannot build {path}: {e}") from e
            if not _build.is_fresh():
                raise NativeError(f"{path} was built from different sources (build.sha256 does not match csrc/ and "
                                  f"include/) and rebuilding failed: {e}") from e
    if not os.path.exists(path):
        raise NativeError(f"{path} is missing; run `python -m coda_b200.build`")
    if os.environ.get("CODA_B200_NO_BUILD") and not _build.is_fresh():
        sys.stderr.write(f"coda_b200: WARNING: {path} does not match the current sources (CODA_B200_NO_BUILD is set)\n")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError here == header/library drift
        fn.restype = res
        fn.argtypes = args
    if lib.coda_b200_version() != VERSION:
        raise NativeError(f"{path} reports ABI version {lib.coda_b200_version()}, this binding expects {VERSION}")
    _LIB = lib
    return lib


def last_error() -> str:
    return load().coda_b200_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != OK:
        raise NativeError(f"coda_b200 {what} failed (rc={rc}): {last_error()}")


def require_device() -> None:
    """Fail loudly if the CUDA path cannot run (no silent CPU route exists)."""
    check(load().coda_b200_device_check(), "device_check")


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)
