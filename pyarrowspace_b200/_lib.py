"""ctypes binding of ``libarrowspace_b200.so`` (the C ABI in ``include/arrowspace_b200.h``).

The library is the product: hand-written sm_100a CUDA behind ``extern "C"`` entry points.
If it is missing or there is no CUDA device every compute call raises -- there is no CPU
fallback and nothing here imports ``oracle/``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ASP_B200_LIB") or os.path.join(_HERE, "libarrowspace_b200.so")   # override: A/B of two builds

ASP_OK = 0
ASP_ERR_EMPTY = 1
ASP_ERR_ZERO_VECTOR = 2
ASP_ERR_LAMBDA_ZERO = 3
ASP_ERR_ARG = 4
ASP_ERR_NOMEM = 5
ASP_ERR_CUDA = 6
ASP_ERR_UNSUPPORTED = 7
ASP_NEED_EXACT = 8
ASP_ERR_LIMIT = 9

GRAM_SEGMENTS = 8
GRAM_SLICES = 24
ROW_UNIT = 32

KERNEL = {"inv_power": 0, "gaussian": 1}
TAU_MODE = {"median": 0, "median_abs": 1, "mean": 2, "fixed": 3}
LAMBDA_FORM = {"bounded": 0, "synthetic": 1}
SYMMETRISE = {"max": 0, "avg": 1, "min": 2, "none": 3}
LAPLACIAN = {"combinatorial": 0, "sym": 1, "rw": 2}
DISTANCE = {"cosine": 0, "l2": 1, "l2sq": 2}

# Named sets of the switches the reference's tests cannot pin (SURVEY.md 8(c)).  "default" is the documented recipe
# (GRAPH_VARIABLES.md:3,7-10; TAUMODE.md:18-19,24-25; SURVEY.md Appendix A); "kat12" is the set that reproduces all 12
# indices of /root/reference/tests/test_0.py:29-61 (DESIGN.md section 1).
PROFILES = {
    "default": {},
    "kat12": {"symmetrise": "none", "laplacian": "sym", "k_counts_self": True, "topk_prunes": True},
}
SWITCH_KEYS = ("kernel", "tau_mode", "tau_fixed", "lambda_form", "symmetrise", "laplacian", "k_counts_self", "topk_prunes",
               "distance", "profile")


class GraphParams(C.Structure):
    _fields_ = [("eps", C.c_double), ("k", C.c_int64), ("topk", C.c_int64), ("p", C.c_double),
                ("sigma", C.c_double), ("has_sigma", C.c_int32)]


class Switches(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("tau_mode", C.c_int32), ("tau_fixed", C.c_double), ("lambda_form", C.c_int32),
                ("symmetrise", C.c_int32), ("laplacian", C.c_int32), ("k_counts_self", C.c_int32),
                ("topk_prunes", C.c_int32), ("distance", C.c_int32)]


class Reduction(C.Structure):
    """asp_reduction (SURVEY.md 8(f)-1): sampler keep rate, seed, cluster count (0 = rule), Lloyd iterations, two-NN probes."""
    _fields_ = [("sample_rate", C.c_double), ("seed", C.c_uint64), ("n_clusters", C.c_int32), ("max_iters", C.c_int32),
                ("probes", C.c_int32), ("reserved", C.c_int32)]


class ReductionInfo(C.Structure):
    _fields_ = [("n_sampled", C.c_int64), ("n_probes", C.c_int64), ("two_nn_mean_ratio", C.c_double),
                ("intrinsic_dim", C.c_int32), ("n_clusters", C.c_int32), ("iters", C.c_int32), ("converged", C.c_int32)]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class LibraryError(RuntimeError):
    """A call into libarrowspace_b200.so failed (code + the library's message)."""

    def __init__(self, code, message):
        super().__init__("%s (arrowspace_b200 error %d)" % (message, code))
        self.code = code
        self.message = message


# name -> (restype, argtypes); every symbol include/arrowspace_b200.h declares
_vp, _i64, _i32, _dbl, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_int
SYMBOLS = {
    "asp_last_error": (C.c_char_p, []),
    "asp_abi_version": (_int, []),
    "asp_default_switches": (None, [C.POINTER(Switches)]),
    "asp_ctx_create": (_int, [_int, C.POINTER(_vp)]),
    "asp_ctx_destroy": (None, [_vp]),
    "asp_ctx_device": (_int, [_vp]),
    "asp_ctx_set_stream": (_int, [_vp, _vp]),
    "asp_ctx_synchronize": (_int, [_vp]),
    "asp_ctx_launch_count": (_i64, [_vp]),
    "asp_build": (_int, [_vp, _vp, _i64, _i32, C.POINTER(GraphParams), C.POINTER(Switches),
                         C.POINTER(_vp), C.POINTER(_vp)]),
    "asp_shard_rows": (_int, [_i64, _int, _int, C.POINTER(_i64), C.POINTER(_i64)]),
    "asp_space_create": (_int, [_vp, _vp, _i64, _i32, _i64, _int, _int, C.POINTER(_vp)]),
    "asp_space_adopt": (_int, [_vp, _vp, _i64, _i32, C.POINTER(_vp)]),
    "asp_space_adopt_shard": (_int, [_vp, _vp, _i64, _i32, _i64, _int, _int, C.POINTER(_vp)]),
    "asp_space_import_lambdas": (_int, [_vp, _vp, _vp]),
    "asp_ctx_trim": (_int, [_vp, C.c_size_t]),
    "asp_space_gram_partials": (_int, [_vp, _vp]),
    "asp_graph_from_gram": (_int, [_vp, _vp, _i32, _i64, C.POINTER(GraphParams), C.POINTER(Switches),
                                   _vp, _vp, _i64, _vp, _i64, C.POINTER(_i64), C.POINTER(_vp)]),
    "asp_space_exact_pairs": (_int, [_vp, _vp, _i64, _vp]),
    "asp_space_compute_lambdas": (_int, [_vp, _vp]),
    "asp_space_dims": (_int, [_vp, C.POINTER(_i64), C.POINTER(_i32), C.POINTER(_i64), C.POINTER(_i64)]),
    "asp_space_lambdas": (_int, [_vp, _vp]),
    "asp_space_norms": (_int, [_vp, _vp]),
    "asp_space_get_item": (_int, [_vp, _i64, _vp, _vp]),
    "asp_space_items": (_int, [_vp, _vp]),
    "asp_graph_info": (_int, [_vp, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(GraphParams)]),
    "asp_graph_csr": (_int, [_vp, _vp, _vp, _vp]),
    "asp_graph_from_csr": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, C.POINTER(GraphParams), C.POINTER(Switches), _int, C.POINTER(_vp)]),
    "asp_graph_switches": (_int, [_vp, C.POINTER(Switches)]),
    "asp_query_lambda": (_int, [_vp, _vp, C.POINTER(Switches), _vp, _i64, _vp, _vp, _vp]),
    "asp_search_batch": (_int, [_vp, _vp, _vp, _i64, _dbl, _vp, _vp, _vp]),
    "asp_search_hybrid_batch": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _vp, _vp, _vp]),
    "asp_hybrid_pool": (_i64, [_i64, _i64, _i64]),
    "asp_search_hybrid_shard": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _vp, _vp, _vp, _vp]),
    "asp_hybrid_merge": (_int, [_vp, _vp, _vp, _vp, _int, _i64, _i64, _i64, _vp, _vp]),
    "asp_search_batch_filtered": (_int, [_vp, _vp, _vp, _i64, _dbl, _vp, _vp, _vp, _vp]),
    "asp_search_hybrid_batch_filtered": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _vp, _vp, _vp, _vp]),
    "asp_search_hybrid_shard_filtered": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _vp, _vp, _vp, _vp, _vp]),
    "asp_search_batch_k": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _vp, _vp, _vp, _vp]),
    "asp_search_batch_taus": (_int, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "asp_search_hybrid_batch_k": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _i64, _vp, _vp, _vp, _vp]),
    "asp_search_hybrid_shard_k": (_int, [_vp, _vp, _vp, _i64, _dbl, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "asp_search_range_batch": (_int, [_vp, _vp, _vp, _i64, _dbl, _dbl, _vp, _i64, _vp, _vp, C.POINTER(_vp)]),
    "asp_range_result_fetch": (_int, [_vp, _vp, _vp]),
    "asp_range_result_free": (None, [_vp]),
    "asp_range_sub_batch": (_i64, []),
    "asp_range_merge": (_int, [_vp, _int, _i64, _vp, _vp, _vp, _vp, _vp]),
    "asp_debug_tc_dots": (_int, [_vp, _vp, _i64, _vp]),
    "asp_topk_merge": (_int, [_vp, _vp, _vp, _int, _i64, _i64, _vp, _vp]),
    "asp_peer_exchange_bytes": (C.c_size_t, [_int, _i64, _i64]),
    "asp_peer_merge": (_int, [_vp, _int, _int, C.POINTER(C.c_uint64), _i64, _i64, _vp, _vp, _i64, _i64, _vp, _vp]),
    "asp_item_graph": (_int, [_vp, C.POINTER(GraphParams), C.POINTER(Switches), C.POINTER(_vp)]),
    "asp_item_knn_rows": (_int, [_vp, C.POINTER(GraphParams), C.POINTER(Switches), _i64, _i64, _vp, _vp, _vp, C.POINTER(_i32)]),
    "asp_graph_from_knn": (_int, [_vp, _i64, _i32, _vp, _vp, _vp, C.POINTER(GraphParams), C.POINTER(Switches), C.POINTER(_vp)]),
    "asp_default_reduction": (None, [C.POINTER(Reduction)]),
    "asp_reduction_sample": (_int, [C.POINTER(Reduction), _i64, _i64, _vp, C.POINTER(_i64)]),
    "asp_space_reduce": (_int, [_vp, C.POINTER(Reduction), _i64, C.POINTER(ReductionInfo), C.POINTER(_vp)]),
    "asp_space_feature_graph": (_int, [_vp, C.POINTER(GraphParams), C.POINTER(Switches), C.POINTER(_vp)]),
    "asp_build_reduced": (_int, [_vp, _vp, _i64, _i32, C.POINTER(GraphParams), C.POINTER(Switches), C.POINTER(Reduction),
                                 C.POINTER(_vp), C.POINTER(_vp), C.POINTER(ReductionInfo), C.POINTER(_vp)]),
    "asp_free_space": (None, [_vp]),
    "asp_free_graph": (None, [_vp]),
    "asp_ctx_stat": (_dbl, [_vp, C.c_char_p]),
}

_lib = None


def load():
    """dlopen the library and type every entry point.  Raises if the .so is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libarrowspace_b200.so is not built (run `python -m pyarrowspace_b200.build`); "
                "arrowspace_b200 has no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != ASP_OK:
        msg = load().asp_last_error()
        raise LibraryError(rc, msg.decode("utf-8", "replace") if msg else "unknown error")


_contexts = {}


def context(device=None):
    """One asp_ctx per (process, device).  Fails loudly without a CUDA device."""
    lib = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _contexts:
        h = _vp()
        check(lib.asp_ctx_create(int(device), C.byref(h)))
        _contexts[device] = h
    return _contexts[device]


def make_params(eps, k, topk, p, sigma):
    return GraphParams(float(eps), int(k), int(topk), float(p), float(sigma if sigma is not None else 0.0),
                       0 if sigma is None else 1)


def make_switches(kernel="inv_power", tau_mode="median", tau_fixed=0.0, lambda_form="bounded", symmetrise="max",
                  laplacian="combinatorial", k_counts_self=False, topk_prunes=False, distance="cosine", profile=None):
    if profile is not None:
        kw = dict(kernel=kernel, tau_mode=tau_mode, tau_fixed=tau_fixed, lambda_form=lambda_form, symmetrise=symmetrise,
                  laplacian=laplacian, k_counts_self=k_counts_self, topk_prunes=topk_prunes, distance=distance)
        kw.update(PROFILES[profile])
        return make_switches(**kw)
    return Switches(KERNEL[kernel], TAU_MODE[tau_mode], float(tau_fixed), LAMBDA_FORM[lambda_form], SYMMETRISE[symmetrise],
                    LAPLACIAN[laplacian], int(bool(k_counts_self)), int(bool(topk_prunes)), DISTANCE[distance])


def make_reduction(reduction):
    """asp_reduction from the `reduction=` extra: True -> the defaults (keep rate 0.6, seed 42, K by rule, 10 Lloyd
    iterations, 2048 two-NN probes); a dict overrides single fields."""
    red = Reduction()
    load().asp_default_reduction(C.byref(red))
    if isinstance(reduction, dict):
        known = {name for name, _ in Reduction._fields_} - {"reserved"}
        for key, val in reduction.items():
            if key not in known:
                raise ValueError("unknown reduction option %r (known: %s)" % (key, ", ".join(sorted(known))))
            setattr(red, key, val)
    elif reduction is not True:
        raise TypeError("reduction= expects True or a dict of options")
    return red


def switches_from(extras):
    """asp_switches from the keyword-only extras of the build entry points (unknown keys are left to the caller)."""
    return make_switches(**{k: extras[k] for k in SWITCH_KEYS if k in extras})
