"""ctypes binding of libfrender_b200.so (include/frender_b200.h).

There is no CPU fallback: importing this module without the built library, or
creating a context without a B200, raises.  Build with `python -m frender_b200.build`
(or `__graft_entry__.build()`).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfrender_b200.so")

OK = 0
ERR_CUDA, ERR_ARG, ERR_BAD_HEADER, ERR_BAD_ALPHABET, ERR_KEY_TOO_LONG = -1, -2, -3, -4, -5
ERR_TABLE_FULL, ERR_BAD_LENGTH, ERR_KEY_NOT_FOUND, ERR_NCCL, ERR_IO, ERR_STATE = -6, -7, -8, -9, -10, -11
RULE_SCAN, RULE_DEMUX = 0, 1
CARRY = 0xFFFFFFFFFFFFFFFF
K_SCAN, K_EXPORT, K_MATCH, K_ROUTE, K_OTHER, K_VERIFY, K_INFLATE = range(7)
K_NUM = 7
READ_TYPES = ("undetermined", "index_hop", "demuxable", "ambiguous")

u64, u32, i32, u8 = C.c_uint64, C.c_uint32, C.c_int32, C.c_uint8
P = C.POINTER
vp = C.c_void_p

# name -> (restype, argtypes); the test-suite checks this list against the header
SIGNATURES = {
    "frb_version": (C.c_int, []),
    "frb_device_count": (C.c_int, [P(C.c_int)]),
    "frb_create": (C.c_int, [C.c_int, u32, P(vp)]),
    "frb_destroy": (None, [vp]),
    "frb_last_error": (C.c_char_p, [vp]),
    "frb_sync": (C.c_int, [vp]),
    "frb_host_alloc": (C.c_int, [P(vp), C.c_size_t]),
    "frb_host_free": (C.c_int, [vp]),
    "frb_dev_alloc": (C.c_int, [vp, C.c_size_t, P(vp)]),
    "frb_dev_free": (C.c_int, [vp, vp]),
    "frb_h2d": (C.c_int, [vp, vp, vp, C.c_size_t]),
    "frb_d2h": (C.c_int, [vp, vp, vp, C.c_size_t]),
    "frb_mem_info": (C.c_int, [vp, P(u64), P(u64)]),
    "frb_write_scan_csv": (C.c_int, [C.c_char_p, vp, vp, vp, vp, vp, vp, vp, u64, vp, vp, vp, u32, C.c_int]),
    "frb_pack_key": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, P(u64)]),
    "frb_unpack_key": (C.c_int, [u64, C.c_char_p]),
    "frb_pack_key2": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, P(u64), P(u64)]),
    "frb_unpack_key2": (C.c_int, [u64, u64, C.c_char_p]),
    "frb_write_scan_csv2": (C.c_int, [C.c_char_p, vp, vp, vp, vp, vp, vp, vp, vp, u64, vp, vp, vp, u32, C.c_int]),
    "frb_set_key_width": (C.c_int, [vp, u32]),
    "frb_file_export_hi": (C.c_int, [vp, u32, vp, u64]),
    "frb_total_export_hi": (C.c_int, [vp, vp, u64]),
    "frb_total_load2": (C.c_int, [vp, vp, vp, vp, u64]),
    "frb_sheet_load2": (C.c_int, [vp, vp, vp, vp, vp, vp, u32, u32, u32]),
    "frb_route_load2": (C.c_int, [vp, vp, vp, vp, u64, u32]),
    "frb_scan_begin": (C.c_int, [vp, u32, u64]),
    "frb_scan_chunk_host": (C.c_int, [vp, vp, u64, u64, C.c_int]),
    "frb_scan_chunk_dev": (C.c_int, [vp, vp, u64, u64, C.c_int, vp, vp]),
    "frb_scan_end": (C.c_int, [vp, P(u64), P(u64)]),
    "frb_scan_gz": (C.c_int, [vp, C.c_char_p, u32, u64, P(u64), P(u64), P(u64)]),
    "frb_scan_gz_batch": (C.c_int, [vp, vp, vp, u32, vp, vp, vp, P(C.c_int)]),
    "frb_gz_inflate": (C.c_int, [vp, C.c_char_p, vp, u64, P(u64), P(C.c_int)]),
    "frb_file_count": (C.c_int, [vp, P(u32)]),
    "frb_file_size": (C.c_int, [vp, u32, P(u64), P(u64)]),
    "frb_file_export": (C.c_int, [vp, u32, vp, vp, vp, u64]),
    "frb_total_finish": (C.c_int, [vp, P(u64)]),
    "frb_total_export": (C.c_int, [vp, vp, vp, vp, u64]),
    "frb_total_load": (C.c_int, [vp, vp, vp, u64]),
    "frb_total_merge": (C.c_int, [vp, vp, vp, vp, u64]),
    "frb_reset": (C.c_int, [vp]),
    "frb_resize_tables": (C.c_int, [vp, u32]),
    "frb_sheet_load": (C.c_int, [vp, vp, vp, vp, u32, u32, u32]),
    "frb_match": (C.c_int, [vp, u32, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "frb_demux_ok": (C.c_int, [vp, vp, u32, vp, vp, vp, vp, vp, P(i32)]),
    "frb_route_load": (C.c_int, [vp, vp, vp, u64, u32]),
    "frb_route_pair": (C.c_int, [vp, vp, u64, vp, u64, C.c_int, vp, vp, vp, vp, P(u64), P(u64), P(u64), P(u64)]),
    "frb_route_reset": (C.c_int, [vp]),
    "frb_route_reserve": (C.c_int, [vp, u64]),
    "frb_route_push": (C.c_int, [vp, vp, u64, vp, u64, C.c_int]),
    "frb_route_pop": (C.c_int, [vp, P(vp), P(vp), vp, vp, P(u64), P(u64), P(u64), P(u64)]),
    "frb_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "frb_nccl_init": (C.c_int, [vp, C.c_char_p, C.c_int, C.c_int]),
    "frb_allmerge": (C.c_int, [vp, P(u64)]),
    "frb_shardmerge": (C.c_int, [vp, P(u64)]),
    "frb_allreduce_u64": (C.c_int, [vp, vp, u64]),
    "frb_synth_load": (C.c_int, [vp, u64, u32, u32, u32, vp, vp, vp, u32, u32, u32, u32, u64, u64]),
    "frb_synth_generate": (C.c_int, [vp, u64, u64, C.c_int, vp, u64, P(u64)]),
    "frb_timer_start": (C.c_int, [vp]),
    "frb_timer_stop": (C.c_int, [vp, P(C.c_float)]),
    "frb_prof_enable": (C.c_int, [vp, C.c_int]),
    "frb_prof_read": (C.c_int, [vp, C.c_int, P(C.c_double), P(u64), C.c_int]),
    "frb_launch_count": (u64, [vp]),
}


class FrbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"frender_b200 error {code}: {message}")
        self.code = code
        self.message = message


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m frender_b200.build`. "
            "frender_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()


def check(ctx, rc):
    if rc != OK:
        msg = lib.frb_last_error(ctx)
        raise FrbError(rc, msg.decode(errors="replace") if msg else "")
    return rc
