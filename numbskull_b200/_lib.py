"""ctypes binding of ``libnumbskull_b200.so`` (C ABI: include/numbskull_b200.h).

The library is the only implementation of the hot path: if it is missing or
no CUDA device is present the calls raise -- there is no CPU fallback.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_PKG, "libnumbskull_b200.so")
_lib = None

NB_OK, NB_ERR_INVALID, NB_ERR_NOT_IMPLEMENTED, NB_ERR_CUDA, NB_ERR_UNSUPPORTED, NB_ERR_NOMEM = range(6)


class GraphDesc(C.Structure):
    _fields_ = [
        ("weight", C.c_void_p), ("n_weight", C.c_int64),
        ("variable", C.c_void_p), ("n_variable", C.c_int64),
        ("factor", C.c_void_p), ("n_factor", C.c_int64),
        ("fmap", C.c_void_p), ("n_fmap", C.c_int64),
        ("vmap", C.c_void_p), ("n_vmap", C.c_int64),
        ("factor_index", C.c_void_p), ("n_factor_index", C.c_int64),
        ("device", C.c_int32),
        ("color_seed", C.c_uint64),
        ("global_vid", C.c_void_p),
        ("warp_row_words", C.c_int32),
        ("sigma_shift", C.c_int32),
        ("preset_color", C.c_void_p),
        ("deferred_coloring", C.c_int32),
    ]


class GraphInfo(C.Structure):
    _fields_ = [
        ("n_variable", C.c_int64), ("n_factor", C.c_int64), ("n_weight", C.c_int64),
        ("n_edges", C.c_int64), ("n_colors", C.c_int32), ("wide_headers", C.c_int32),
        ("n_thread_rows", C.c_int64), ("n_warp_rows", C.c_int64), ("stream_words", C.c_int64),
        ("device_bytes", C.c_int64), ("count_entries", C.c_int64), ("jp_rounds", C.c_int64),
        ("max_arity", C.c_int64), ("n_pair_rows", C.c_int64), ("n_fast_rows", C.c_int64),
        ("n_cat_rows", C.c_int64), ("tt_quads", C.c_int64), ("tt2_quads", C.c_int64),
        ("value_bytes", C.c_int32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


# name -> (restype, argtypes); every symbol include/numbskull_b200.h declares
_P, _I64, _I32, _U64, _DBL = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_double
SIGNATURES = {
    "nb_last_error": (C.c_char_p, []),
    "nb_abi_version": (C.c_int, []),
    "nb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "nb_assign_vtf_offsets": (C.c_int, [_P, _I64, C.POINTER(_I64)]),
    "nb_compute_var_map": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _P, _I64]),
    "nb_load_weights": (C.c_int, [_P, _I64, _I64, _P]),
    "nb_load_variables": (C.c_int, [_P, _I64, _I64, _P]),
    "nb_load_domains": (C.c_int, [_P, _I64, _P, _P, _I64, _P, _I64]),
    "nb_load_factors": (C.c_int, [_P, _I64, _I64, _P, _P, _I64, _P, _P, _I64, _P, _I64]),
    "nb_synth_kbc": (C.c_int, [_I64, _U64, _I64, _DBL, _I64, _DBL, _DBL, _DBL, _P, _P, _P, _P, _I64, _P, _I64]),
    "nb_synth_kbc_weights": (C.c_int, [_U64, _I64, _DBL, _P]),
    "nb_synth_kbc_variables": (C.c_int, [_U64, _DBL, _P, _I64, _P]),
    "nb_synth_kbc_block": (C.c_int, [_I64, _U64, _I64, _I64, _DBL, _DBL, _P, _I64, _I64, _P, C.POINTER(_I64), _P,
                                     C.POINTER(_I64)]),
    "nb_block_ghosts": (C.c_int, [_P, _I64, _I64, _I64, _I64, _P, C.POINTER(_I64), C.c_int]),
    "nb_extract_local": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, C.c_int32, C.POINTER(_I64), C.POINTER(_I64),
                                   C.POINTER(_I64), C.POINTER(_I64), _P, _P, _P]),
    "nb_graph_create": (C.c_int, [C.POINTER(GraphDesc), C.POINTER(_P)]),
    "nb_graph_destroy": (None, [_P]),
    "nb_graph_get_info": (C.c_int, [_P, C.POINTER(GraphInfo)]),
    "nb_graph_get_colors": (C.c_int, [_P, _P]),
    "nb_graph_check_coloring": (C.c_int, [_P, C.POINTER(_I64)]),
    "nb_graph_color_edges": (C.c_int, [_P, _P]),
    "nb_set_var_values": (C.c_int, [_P, C.c_int, _P]),
    "nb_get_var_values": (C.c_int, [_P, C.c_int, _P]),
    "nb_set_weights": (C.c_int, [_P, _P]),
    "nb_get_weights": (C.c_int, [_P, _P]),
    "nb_get_weights_dev": (C.c_int, [_P, _P]),
    "nb_set_weights_dev": (C.c_int, [_P, _P]),
    "nb_reset_counts": (C.c_int, [_P]),
    "nb_get_counts": (C.c_int, [_P, _P, C.c_int]),
    "nb_get_counts_marginals": (C.c_int, [_P, _P, C.c_int, _P, _DBL]),
    "nb_get_marginals": (C.c_int, [_P, _P, _DBL]),
    "nb_get_counts_compact": (C.c_int, [_P, _P, _I64, C.POINTER(_I32)]),
    "nb_set_counts": (C.c_int, [_P, _P]),
    "nb_host_alloc": (C.c_int, [C.POINTER(_P), _I64]),
    "nb_host_free": (C.c_int, [_P]),
    "nb_potentials": (C.c_int, [_P, C.c_int, _P, _I64, _P, _P, _I64]),
    "nb_potentials_records": (C.c_int, [_P, C.c_int, _P, _I64, _P, _P, _I64, _P]),
    "nb_gibbs_sweeps": (C.c_int, [_P, _I64, C.c_int, C.c_int, _U64]),
    "nb_learn_sweeps": (C.c_int, [_P, _I64, C.POINTER(_DBL), _DBL, C.c_int, _DBL, _DBL, C.c_int, _U64, _I64]),
    "nb_timer_start": (C.c_int, [_P]),
    "nb_timer_stop": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "nb_synchronize": (C.c_int, [_P]),
    "nb_launch_count": (C.c_int, [_P, C.POINTER(_I64)]),
    "nb_flush_l2": (C.c_int, [_P, _I64]),
    "nb_gibbs_color_phase": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _U64, _I64]),
    "nb_gather_values_dev": (C.c_int, [_P, C.c_int, _P, _I64, _P]),
    "nb_scatter_values_dev": (C.c_int, [_P, C.c_int, _P, _I64, _P]),
    "nb_learn_color_phase": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _DBL, C.c_int, _DBL, _DBL, C.c_int, _U64, _I64]),
    "nb_learn_blocks": (C.c_int, [_P, _DBL, C.c_int, _I64, C.POINTER(C.c_int)]),
    "nb_learn_cell_ids": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, C.POINTER(_I64)]),
    "nb_color_round": (C.c_int, [_P, C.POINTER(_I64)]),
    "nb_color_restart": (C.c_int, [_P, C.c_int]),
    "nb_split_colors": (C.c_int, [_P, _P, _I64]),
    "nb_color_natural_round_cap": (C.c_int, []),
    "nb_gather_colors_dev": (C.c_int, [_P, _P, _I64, _P]),
    "nb_scatter_colors_dev": (C.c_int, [_P, _P, _I64, _P]),
    "nb_color_min_ids": (C.c_int, [_P, C.c_int, _P]),
    "nb_relabel_colors": (C.c_int, [_P, _P, C.c_int]),
    "nb_graph_finalize": (C.c_int, [_P]),
    "nb_p2p_export": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "nb_p2p_open": (C.c_int, [_P, _P, _P, C.c_int]),
    "nb_p2p_local_slots": (C.c_int, [_P, _P, _I64, _P]),
    "nb_p2p_set_plan": (C.c_int, [_P, C.c_int, _P, _P, _P, _P]),
    "nb_p2p_exchange": (C.c_int, [_P, C.c_int, C.c_int]),
    "nb_p2p_wait": (C.c_int, [_P]),
    "nb_gibbs_sweeps_p2p": (C.c_int, [_P, _I64, C.c_int, C.c_int, _U64, C.c_int, C.c_int]),
    "nb_p2p_check": (C.c_int, [_P]),
    "nb_p2p_close": (C.c_int, [_P]),
    "nb_set_stream": (C.c_int, [_P, _P]),
    "nb_begin_epoch": (C.c_int, [_P, C.POINTER(_I64)]),
}


def build(force=False, verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    csrc = os.path.join(_PKG, "csrc")
    cmd = ["make", "-C", csrc, "-j8"] + (["-B"] if force else [])
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("building libnumbskull_b200.so failed")
    return SO_PATH


def lib():
    """The loaded library; raises if it was never built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                "numbskull_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C numbskull_b200/csrc`. There is no CPU fallback." % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.nb_abi_version() != 1:
            raise RuntimeError("libnumbskull_b200.so ABI version mismatch")
        _lib = L
    return _lib


def last_error():
    return lib().nb_last_error().decode("utf-8", "replace")


def check(rc):
    """Translate a status code into the exception the reference would raise."""
    if rc == NB_OK:
        return
    msg = last_error()
    if rc == NB_ERR_NOT_IMPLEMENTED:
        print(msg)  # inference.py:410-412 prints before raising
        raise NotImplementedError("Factor function is not implemented.")
    if rc == NB_ERR_INVALID:
        raise ValueError(msg)
    if rc == NB_ERR_NOMEM:
        raise MemoryError(msg)
    if rc == NB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def device_count():
    n = C.c_int(0)
    rc = lib().nb_device_count(C.byref(n))
    return n.value if rc == NB_OK else 0


def contiguous(a, dtype):
    a = np.asarray(a)
    if a.dtype != dtype or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=dtype)
    return a
