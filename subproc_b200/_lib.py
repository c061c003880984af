"""ctypes binding of libothello_b200.so (include/othello_b200.h).

The CUDA library is the product: there is no Python/CPU fallback.  ``lib()`` raises when the
shared object is missing (it is built in-tree by ``python -m subproc_b200.build``), and every
entry point raises ``OthelloError`` on a non-zero return code.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libothello_b200.so")

ABI_VERSION = 4

u64p = ctypes.POINTER(ctypes.c_uint64)
u8p = ctypes.POINTER(ctypes.c_uint8)
i32p = ctypes.POINTER(ctypes.c_int32)
f32p = ctypes.POINTER(ctypes.c_float)
f64p = ctypes.POINTER(ctypes.c_double)
vp = ctypes.c_void_p
i64 = ctypes.c_int64
i32 = ctypes.c_int32


class PlayoutArgs(ctypes.Structure):
    """othello_playout_args (include/othello_b200.h)."""
    _fields_ = [
        ("seed", ctypes.c_uint64), ("gid0", ctypes.c_uint64), ("n_games", i64),
        ("black0", vp), ("white0", vp), ("turn0", vp),
        ("policy", i32), ("random_plies", i32), ("n_rand_black", i32), ("n_rand_white", i32),
        ("weights", vp), ("t_max", i32), ("stride", i64),
        ("traj_black", vp), ("traj_white", vp), ("traj_move", vp),
        ("nplies", vp), ("final_black", vp), ("final_white", vp),
        ("policy_white", i32), ("games_per_warp", i32), ("weights_white", vp), ("totals", vp), ("summary", vp),
    ]


class PositionInfo(ctypes.Structure):
    """othello_position_info (include/othello_b200.h)."""
    _fields_ = [
        ("black", ctypes.c_uint64), ("white", ctypes.c_uint64), ("flips", ctypes.c_uint64),
        ("legal_black", ctypes.c_uint64), ("legal_white", ctypes.c_uint64),
        ("ret", i32), ("n_black", i32), ("n_white", i32), ("n_empty", i32),
        ("features_black", i32 * 10), ("features_white", i32 * 10),
    ]


# name -> (restype, argtypes); also the export list checked by tests/test_boundary.py
SIGNATURES = {
    "othello_abi_version": (ctypes.c_int, []),
    "othello_error_string": (ctypes.c_char_p, [ctypes.c_int]),
    "othello_legal": (ctypes.c_int, [vp, vp, vp, i64, vp]),
    "othello_flips": (ctypes.c_int, [vp, vp, vp, vp, i64, vp]),
    "othello_step": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]),
    "othello_counts": (ctypes.c_int, [vp, vp, vp, i64, vp]),
    "othello_mask_count": (ctypes.c_int, [vp, vp, vp, vp, vp, i64, vp]),
    "othello_serialize_boards": (ctypes.c_int, [vp, vp, vp, i64, vp]),
    "othello_deserialize_boards": (ctypes.c_int, [vp, vp, vp, i64, vp]),
    "othello_features": (ctypes.c_int, [vp, vp, vp, vp, i64, vp]),
    "othello_eval": (ctypes.c_int, [vp, vp, vp, vp, vp, i64, vp]),
    "othello_playout": (ctypes.c_int, [ctypes.POINTER(PlayoutArgs), vp]),
    "othello_perft_workspace_bytes": (i64, [ctypes.c_int]),
    "othello_perft": (ctypes.c_int, [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, vp, i64,
                                     u64p, vp]),
    "othello_perft_async": (ctypes.c_int, [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, vp, i64, vp, vp]),
    "othello_solve_workspace_bytes": (i64, []),
    "othello_solve": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, i64, vp, i64, vp]),
    "othello_learn_accumulate": (ctypes.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, vp, vp, vp]),
    "othello_learn_stats": (ctypes.c_int, [vp, vp, vp]),
    "othello_learn_refit": (ctypes.c_int, [vp, i32, vp, vp, vp, vp, vp, vp]),
    "othello_learn_solve": (ctypes.c_int, [vp, vp, vp, vp, vp, vp]),
    "othello_value_records": (ctypes.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, vp]),
    "othello_sort_workspace_bytes": (i64, [i64]),
    "othello_sort_records": (ctypes.c_int, [vp, vp, vp, vp, i64, i32, vp, i64, vp]),
    "othello_partition_records": (ctypes.c_int, [vp, vp, vp, vp, i64, i32, vp, vp, i64, vp]),
    "othello_table_workspace_bytes": (i64, [i64]),
    "othello_table_probe": (ctypes.c_int, [vp, i64, vp, vp, i32, vp, i64, vp, vp]),
    "othello_table_apply": (ctypes.c_int, [vp, vp, i64, ctypes.c_double, vp, vp, i32, vp, vp, i64, vp, vp]),
    "othello_table_rehash": (ctypes.c_int, [vp, i64, vp, vp, i32, vp]),
    "othello_table_lookup": (ctypes.c_int, [vp, i64, vp, vp, i32, vp, vp]),
    "othello_unpack_keys": (ctypes.c_int, [vp, vp, i64, vp]),
    "othello_int32_peak_kernel": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "othello_int32_dual_peak_kernel": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "othello_ctx_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(vp)]),
    "othello_ctx_destroy": (None, [vp]),
    "othello_board_apply_host": (ctypes.c_int, [vp, ctypes.c_uint64, ctypes.c_uint64, i32, i32,
                                                ctypes.POINTER(PositionInfo)]),
    "othello_legal_host": (ctypes.c_int, [vp, vp, vp, vp, i64]),
    "othello_step_host": (ctypes.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64]),
    "othello_playout_host": (ctypes.c_int, [vp, ctypes.c_uint64, ctypes.c_uint64, i64, vp, vp, vp, i32, i32, i32, i32,
                                            vp, i32, vp, i32, vp, vp, vp, vp, vp, vp]),
    "othello_playout_host_async": (ctypes.c_int, [vp, ctypes.c_uint64, ctypes.c_uint64, i64, vp, vp, vp, i32, i32, i32,
                                                  i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp,
                                                  ctypes.POINTER(i64)]),
    "othello_ctx_wait": (ctypes.c_int, [vp, i64]),
    "othello_ctx_set_option": (ctypes.c_int, [vp, i32, i64]),
    "othello_ctx_trajectory": (ctypes.c_int, [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp),
                                              ctypes.POINTER(i64), ctypes.POINTER(i32)]),
}


class OthelloError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        msg = _lib.othello_error_string(code).decode() if _lib is not None else "?"
        super().__init__("%s failed: %s (code %d)" % (where, msg, code))


_lib = None


def lib():
    """The loaded library.  Raises (loudly) if it was never built -- there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.isfile(SO):
            raise RuntimeError(
                "subproc_b200: %s is missing -- build it with `python -m subproc_b200.build` "
                "(nvcc, sm_100a). There is no CPU fallback." % SO)
        L = ctypes.CDLL(SO)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        got = L.othello_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError("libothello_b200.so ABI %d != binding ABI %d: rebuild" % (got, ABI_VERSION))
        _lib = L
    return _lib


def check(code, where):
    if code != 0:
        raise OthelloError(code, where)
