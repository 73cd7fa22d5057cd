"""ctypes binding of libhole_b200.so (the C ABI declared in include/hole_b200.h).

There is no fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HOLE_B200_LIB", os.path.join(_HERE, "libhole_b200.so"))   # override: A/B experiments

HOLE_SIDE_TAIL, HOLE_SIDE_HEAD, HOLE_SIDE_BOTH, HOLE_SIDE_RELATION = 0, 1, 2, 3
HOLE_RANK_BF16, HOLE_RANK_BF16X3 = 0, 1
HOLE_OPT_SGD, HOLE_OPT_ADAGRAD = 0, 1
ABI_VERSION = 7


class HoleError(RuntimeError):
    pass


_p, _i64, _i32, _u64, _f32, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_float, C.c_int

#: name -> (restype, argtypes); kept in step with include/hole_b200.h (tests check it)
SIGNATURES = {
    "hole_abi_version": (_int, []),
    "hole_last_error": (C.c_char_p, []),
    "hole_row_stride": (_int, [_int]),
    "hole_ctx_create": (_int, [C.POINTER(_p), _int, _i64, _int]),
    "hole_ctx_destroy": (_int, [_p]),
    "hole_ctx_set_relations": (_int, [_p, _i64]),
    "hole_ctx_set_score_mode": (_int, [_p, _int]),
    "hole_ctx_set_optimizer": (_int, [_p, _int, _p]),
    "hole_pack_rows": (_int, [_p, _p, _p, _i64, _p]),
    "hole_unpack_rows": (_int, [_p, _p, _p, _i64, _p]),
    "hole_corrupt": (_int, [_p, _p, _i64, _p, _p, _p, _u64, _u64, _p, _p, C.POINTER(_int), _p]),
    "hole_corrupt_at": (_int, [_p, _p, _i64, _p, _p, _p, _u64, _u64, _u64, _p, _p, C.POINTER(_int), _p]),
    "hole_score": (_int, [_p, _p, _p, _i64, _p, _p]),
    "hole_train_step": (_int, [_p, _p, _p, _p, _int, _i64, _f32, _f32, _p, _p, _p]),
    "hole_train_step_ex": (_int, [_p, _p, _p, _p, _p, _int, _i64, _f32, _f32, _p, _p, _p]),
    "hole_train_step_plan": (_int, [_p, _p, _p, _i64, _p]),
    "hole_train_step_logloss": (_int, [_p, _p, _p, _p, _i64, _int, _p, _p, _p, _u64, _u64, _f32, _f32, _p, _p, _p, _p, _p]),
    "hole_shard_route": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p, _p, _p, _p, _p]),
    "hole_shard_post": (_int, [_p, _p, _p, _int, _int, _i64, _p, _p, _p]),
    "hole_shard_init": (_int, [_p, _int, _int, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, C.c_double,
                                _p, _p, _p]),
    "hole_shard_prepare": (_int, [_p, _p, _i64, _u64, _u64, _p]),
    "hole_shard_step": (_int, [_p, _p, _i64, _u64, _u64, _f32, _f32, _p, _p]),
    "hole_shard_step_compute": (_int, [_p, _p, _i64, _u64, _u64, _f32, _f32, _p, _p]),
    "hole_shard_step_apply": (_int, [_p, _p]),
    "hole_shard_steps": (_int, [_p, _p, _i64, _i64, _u64, _u64, _f32, _p, _p, _p]),
    "hole_shard_steps_host": (_int, [_p, _p, _i64, _i64, _u64, _u64, _f32, _p, _p, _p]),
    "hole_shard_poll": (_int, [_p, C.POINTER(_int), _p]),
    "hole_shard_set_optimizer": (_int, [_p, _int, _p]),
    "hole_shard_step_logloss": (_int, [_p, _p, _i64, _int, _u64, _u64, _f32, _f32, _p, _p, _p, _p, _p]),
    "hole_shard_step_logloss_compute": (_int, [_p, _p, _i64, _int, _u64, _u64, _f32, _f32, _p, _p, _p, _p, _p]),
    "hole_shard_profile_read": (_int, [_p, C.POINTER(C.c_double), C.POINTER(_i64)]),
    "hole_enable_peer_access": (_int, [_p, _int]),
    "hole_gather_rows": (_int, [_p, _p, _p, _i64, _p, _i64, _p]),
    "hole_add_rows": (_int, [_p, _p, _p, _i64, _p, _i64, _p]),
    "hole_train_steps": (_int, [_p, _p, _p, _i64, _i64, _p, _p, _p, _u64, _u64, _f32, _p, _p, _p, _p]),
    "hole_train_steps_host": (_int, [_p, _p, _p, _i64, _i64, _p, _p, _p, _u64, _u64, _f32, _p, _p, _p]),
    "hole_rank": (_int, [_p, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, _int, _p, _p, _p]),
    "hole_rank_ex": (_int, [_p, _p, _i64, _i64, _p, _p, _i64, _int, _int, _p, _p, _p, _int, _p, _p, _p]),
    "hole_rank_prepare": (_int, [_p, _p, _i64, _i64, _int, _p]),
    "hole_rank_invalidate": (_int, [_p]),
    "hole_topk": (_int, [_p, _p, _i64, _i64, _p, _i64, _int, _int, _int, _p, _p, _p, _p, _p]),
    "hole_neighbors": (_int, [_p, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, _p, _p]),
    "hole_rank_typed": (_int, [_p, _p, _p, _i64, _int, _int, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p]),
    "hole_topk_typed": (_int, [_p, _p, _p, _p, _i64, _int, _int, _int, _p, _p, _i64, _p, _p, _p, _p, _p]),
    "hole_rank_debug_operands": (_int, [_p, _p, _p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_int), _p]),
    "hole_profile_enable": (_int, [_p, _int]),
    "hole_profile_read": (_int, [_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_i64)]),
    "hole_parse_triples": (_i64, [C.c_char_p, _p, _i64]),
    "hole_crc32c": (C.c_uint32, [C.c_uint32, _p, _u64]),
    "hole_launch_count": (_i64, []),
    "hole_launch_count_reset": (None, []),
}

_lib = None


def load():
    """Load the shared library (once).  Raises HoleError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HoleError(
            f"{LIB_PATH} not found: build it with `python -m graphembeddings_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.hole_abi_version() != ABI_VERSION:
        raise HoleError(f"ABI mismatch: library {lib.hole_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().hole_last_error().decode("utf-8", "replace")
        raise HoleError(f"libhole_b200 error {rc}: {msg}")
