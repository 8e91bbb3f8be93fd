"""ctypes binding of libdiskann_b200.so — the C ABI declared in include/diskann_b200.h.

There is no CPU fallback: if the shared library is missing or cannot be loaded this module
raises, and every entry point that needs a GPU fails with DAB_ERR_NO_DEVICE when none is
visible.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DAB_LIB_PATH") or os.path.join(_HERE, "libdiskann_b200.so")  # override: another build of the library (A/B)

# every symbol include/diskann_b200.h declares: name -> (restype, argtypes)
_vp, _u32, _u64, _i, _f = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int, C.c_float
SYMBOLS = {
    "dab_create": (_i, [C.POINTER(_vp), _i, _i, _u32, _u64, _u32, _u32, _i]),
    "dab_destroy": (None, [_vp]),
    "dab_last_error": (C.c_char_p, []),
    "dab_set_stream": (_i, [_vp, _vp]),
    "dab_launch_count": (_u64, []),
    "dab_upload_vectors": (_i, [_vp, _vp, _u64, _u64]),
    "dab_upload_vectors_device": (_i, [_vp, _vp, _u64, _u64]),
    "dab_upload_graph": (_i, [_vp, _vp, _u32, _u64, _u64]),
    "dab_upload_graph_device": (_i, [_vp, _vp, _u32, _u64, _u64]),
    "dab_download_graph": (_i, [_vp, _vp, _u32, _u64, _u64]),
    "dab_upload_pq": (_i, [_vp, _vp, _u32, _vp, _u32, _vp]),
    "dab_pq_train": (_i, [_vp, _vp, _u64, _u32, _u32, _u32, _u64]),
    "dab_pq_encode_all": (_i, [_vp]),
    "dab_pq_download": (_i, [_vp, _vp, _vp, _vp]),
    "dab_comm_unique_id": (_i, [_vp]),
    "dab_comm_init": (_i, [_vp, _vp, _i, _i]),
    "dab_broadcast_index": (_i, [_vp, _i]),
    "dab_comm_destroy": (_i, [_vp]),
    "dab_broadcast": (_i, [_vp, _i]),
    "dab_pair_distances": (_i, [_i, _i, _i, _u32, _vp, _vp, _u64, _vp, _i]),
    "dab_distances": (_i, [_vp, _vp, _u32, _vp, _u32, _vp]),
    "dab_distances_device": (_i, [_vp, _vp, _u32, _vp, _u32, _vp]),
    "dab_row_pair_distances": (_i, [_vp, _vp, _vp, _u64, _vp]),
    "dab_pairwise": (_i, [_vp, _vp, _u32, _vp]),
    "dab_search_batch": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "dab_search_batch_device": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "dab_search_batch_async": (_i, [_vp, _u32, _vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "dab_search_batch_device_async": (_i, [_vp, _u32, _vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "dab_wait": (_i, [_vp, _u32]),
    "dab_pq_populate_lut": (_i, [_vp, _vp, _u32, _i, _vp]),
    "dab_pq_distances": (_i, [_vp, _vp, _u32, _vp, _u32, _vp]),
    "dab_pq_encode": (_i, [_vp, _vp, _u64, _vp]),
    "dab_pq_self_distances": (_i, [_vp, _vp, _vp, _u64, _vp]),
    "dab_search_batch_pq": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "dab_search_batch_pq_rerank": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "dab_search_batch_pq_device": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _i, _vp, _vp, _vp, _vp, _vp]),
    "dab_sq_compress": (_i, [_i, _vp, _f, _u32, _i, _vp, _u64, _vp, _vp]),
    "dab_sq_distances": (_i, [_i, _i, _i, _f, _f, _u32, _vp, _vp, _vp, _vp, _u64, _vp]),
    "dab_upload_sq": (_i, [_vp, _i, _vp, _f, _f, _f, _vp]),
    "dab_sq_encode_all": (_i, [_vp]),
    "dab_sq_download": (_i, [_vp, _vp]),
    "dab_search_batch_sq": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _i, _vp, _vp, _vp, _vp, _vp]),
    "dab_search_batch_sq_device": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _i, _vp, _vp, _vp, _vp, _vp]),
    "dab_minmax_row_bytes": (_u32, [_u32, _i]),
    "dab_minmax_compress": (_i, [_i, _f, _u32, _i, _vp, _u64, _vp, _vp]),
    "dab_minmax_distances": (_i, [_i, _i, _i, _i, _u32, _vp, _vp, _u64, _vp]),
    "dab_minmax_query_distances": (_i, [_i, _i, _i, _u32, _vp, _u32, _vp, _u64, _vp]),
    "dab_robust_prune": (_i, [_vp, _vp, _vp, _vp, _vp, _u32, _u32, _u32, _f, _vp, _vp]),
    "dab_build": (_i, [_vp, _u32, _u32, _f, _u32]),
    "dab_flat_knn": (_i, [_vp, _vp, _u32, _u32, _vp, _vp]),
    "dab_flat_knn_tc": (_i, [_vp, _vp, _u32, _u32, _vp, _vp]),
}

_lib = None


class DabError(RuntimeError):
    """A non-zero status from the C ABI (maps to ANNError in the reference)."""

    def __init__(self, code, message):
        super().__init__(f"diskann_b200 error {code}: {message}")
        self.code = code


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C diskann_b200/csrc). There is no CPU fallback for the product path.")
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(code):
    if code != 0:
        raise DabError(code, lib().dab_last_error().decode("utf-8", "replace"))
