"""ctypes binding of libevz.so (include/evz.h).  There is no fallback: if the CUDA library
is missing the import of the engine fails loudly."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libevz.so")

EVZ_ROW_ALIGN = 256
EVZ_DESC_BYTES = 128
EVZ_MAX_KP = 12288
EVZ_R_MAX = 16383

ST_OK, ST_FEW_MATCHES, ST_FEW_POINTS, ST_NO_MODEL_1, ST_NO_MODEL_2, ST_FEW_INLIERS = 0, 1, 3, 4, 5, 6

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_d = C.c_double

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/evz.h exactly
SIGNATURES = {
    "evz_version": [],
    "evz_create": [_i, C.POINTER(_p)],
    "evz_destroy": [_p],
    "evz_last_error": [_p],
    "evz_sm_count": [_p],
    "evz_set_option": [_p, _i, _i],
    "evz_match_kernel_ms": [_p, _i, C.POINTER(C.c_float)],
    "evz_ingest": [_p, _p, _i, _i, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p],
    "evz_match_top2": [_p, _p, _p, _i64, _p, _p, _p, _p, _p, _i, _p, _p, _p],
    "evz_match_top2_d": [_p, _p, _i, _p, _i64, _p, _p, _p, _p, _p, _i, _p, _p, _p],
    "evz_filter_matches": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _d, _i, _p, _p, _p, _p, _p, _p, _p],
    "evz_find_homography": [_p, _p, _p, _p, _i, _i, _p, _i, C.c_uint32, _i64, _i, _d, _d, _i,
                            _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "evz_find_homography_ids": [_p, _p, _p, _p, _i, _i, _p, _i, C.c_uint32, _p, _i, _d, _d, _i,
                                _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "evz_static_filter": [_p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "evz_concat_dedup": [_p, _i, C.POINTER(_p), C.POINTER(_p), C.POINTER(_p), _i, _p, _i, _p, _p, _p, _p],
    "evz_chain_scan": [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p],
    "evz_chain_scan_segments": [_p, _p, _p, _i, _p, _i, _i, _p, _p, _p],
    "evz_chain_ref_step": [_p, _p, _p, _i, _i, _i, _p, _p, _p, _p],
    "evz_chain_seed_apply": [_p, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "evz_remap": [_p, _p, _p, _i64, _p, _i, _d, _d, _i, _p, _p],
    "evz_max_movement": [_p, _p, _i, _i, _i, _p, _p],
}
_RESTYPES = {"evz_destroy": None, "evz_last_error": C.c_char_p}

_lib = None


class EvzError(RuntimeError):
    pass


def load():
    """Load libevz.so.  Raises ImportError (with the build command) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"or `make -C evenvizion_b200/csrc`.  evenvizion_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, _i)
    _lib = lib
    return lib


def check(handle, rc):
    if rc != 0:
        msg = load().evz_last_error(handle)
        raise EvzError(f"libevz error {rc}: {msg.decode() if msg else ''}")
