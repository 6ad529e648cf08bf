"""ctypes binding of libcalfkit_b200.so (C-ABI: include/calfkit_b200.h).

There is deliberately no fallback: if the CUDA library is missing or cannot be loaded the engine
raises EngineError — the product never routes through a CPU implementation."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from calfkit.exceptions import EngineError

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
LIB_PATH = os.environ.get("CK_LIB") or os.path.join(_PKG_ROOT, "libcalfkit_b200.so")   # CK_LIB: kernel A/B builds during development

# ---- constants mirrored from csrc/ck_common.h (checked against the header in tests/test_abi.py) ----
CK_OK, CK_NOT_CANONICAL, CK_JSON_INVALID, CK_SCHEMA_INVALID, CK_UNSUPPORTED, CK_EMPTY, CK_BAD_FRAME = range(7)
STATUS_NAMES = ["ok", "not_canonical", "json_invalid", "schema_invalid", "unsupported", "empty", "bad_frame"]
(CK_ACT_NONE, CK_ACT_RETURN, CK_ACT_SILENT, CK_ACT_RAISES, CK_ACT_CALL, CK_ACT_TAILCALL, CK_ACT_FANOUT,
 CK_ACT_HOST_TOOL, CK_ACT_REPLY, CK_ACT_GATE_COMPLETE, CK_ACT_GATE_PASS) = range(11)
ACTION_NAMES = ["none", "return", "silent", "raises", "call", "tailcall", "fanout", "host_tool", "reply", "gate_complete", "gate_pass"]

COLS = ["STATUS", "ACTION", "ERR", "CORR_OFF", "CORR_LEN", "NFRAMES", "FRAMES_OFF", "FRAMES_LEN", "TOP_OFF", "TOP_LEN",
        "TGT_OFF", "TGT_LEN", "CB_OFF", "CB_LEN", "NARGS", "ARG0_OFF", "ARG0_LEN", "ARG1_OFF", "ARG1_LEN", "ARGKINDS",
        "FOV_OFF", "FOV_LEN", "TC_OFF", "TC_LEN", "TR_OFF", "TR_LEN", "UNC_OFF", "UNC_LEN", "HIST_OFF", "HIST_LEN",
        "FOP_OFF", "FOP_LEN", "TI_OFF", "TI_LEN", "SMETA_OFF", "SMETA_LEN", "SOV_OFF", "SOV_LEN", "PD_OFF", "PD_LEN",
        "WFMETA_OFF", "WFMETA_LEN", "CALL_VAL_OFF", "CALL_VAL_LEN", "TNAME_OFF", "TNAME_LEN", "ARGS_OFF", "ARGS_LEN",
        "RES_OFF", "RES_LEN", "NOUT", "ODATA_OFF", "ODATA_LEN", "OTEXT_OFF", "OTEXT_LEN"]
COL = {name: i for i, name in enumerate(COLS)}
NUM_COLS = len(COLS)

KERNELS = ["walk", "plan", "scan", "emit", "route", "fanout", "canon", "walk_long", "walk_elems", "codec"]
NUM_KERNELS = len(KERNELS)

PUB_DTYPE = np.dtype([("payload", "<u4"), ("topic_id", "<i4"), ("topic_off", "<u4"), ("topic_len", "<u4"),
                      ("record", "<u4"), ("has_key", "<u4"), ("partition", "<i4"), ("pad", "<u4")])

EXPORTS = ["ck_create", "ck_destroy", "ck_last_error", "ck_version", "ck_register_topics", "ck_set_tool_node", "ck_submit",
           "ck_submit_device", "ck_tool_args", "ck_tool_plan", "ck_tool_plan_device", "ck_return_plan", "ck_set_agent_node", "ck_set_agent_tool_topic_ids", "ck_fanout_plan", "ck_tailcall_plan", "ck_exchange_plan", "ck_launch_count", "ck_reply_plan",
           "ck_sync", "ck_out_size", "ck_fetch_columns", "ck_fetch_output", "ck_fetch_overlay", "ck_fetch_topic_hist", "ck_stream",
           "ck_device_buffers", "ck_device_buffers2", "ck_gather_spans", "ck_profile", "ck_profile_read", "ck_fetch_cols",
           "ck_host_alloc", "ck_host_free", "ck_canon_stats", "ck_fetch_output_async",
           "ck_fetch_cols_async", "ck_gate_create", "ck_gate_register", "ck_gate_arrive", "ck_gate_stats", "ck_gate_reset", "ck_submit_recordbatch",
           "ck_fetch_rb_index", "ck_fetch_rb_decompressed", "ck_encode_recordbatch", "ck_encode_recordbatches", "ck_fetch_recordbatches", "ck_group_publishes", "ck_fetch_groups", "ck_comm_create", "ck_comm_connect", "ck_exchange_send", "ck_recv_info", "ck_fetch_received", "ck_peek_received", "ck_fetch_received_async", "ck_set_option"]

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineError(f"{LIB_PATH} not found: build it with `python calfkit-sdk_b200/build.py` "
                          "(there is no CPU fallback)")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise EngineError(f"cannot load {LIB_PATH}: {e}") from e
    vp, u8p, u32p, i32p, i64p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    sig = {
        "ck_create": (C.c_int, [C.c_int, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(vp)]),
        "ck_destroy": (None, [vp]),
        "ck_last_error": (C.c_char_p, [vp]),
        "ck_version": (C.c_int, []),
        "ck_register_topics": (C.c_int, [vp, u8p, u32p, C.c_uint32, i32p, C.c_uint32]),
        "ck_set_tool_node": (C.c_int, [vp, C.c_int32, C.c_uint32, u32p, u8p, u32p]),
        "ck_submit": (C.c_int, [vp, u8p, i64p, C.c_uint32]),
        "ck_submit_device": (C.c_int, [vp, u8p, i64p, C.c_uint32]),
        "ck_tool_args": (C.c_int, [vp]),
        "ck_tool_plan": (C.c_int, [vp, u8p, i64p]),
        "ck_tool_plan_device": (C.c_int, [vp, u8p, i64p]),
        "ck_return_plan": (C.c_int, [vp]),
        "ck_set_agent_node": (C.c_int, [vp, C.c_int32, u8p, C.c_uint32, u8p, C.c_uint32, u8p, u32p, u8p, u32p, C.c_uint32]),
        "ck_set_agent_tool_topic_ids": (C.c_int, [vp, C.c_int32, u32p, C.c_uint32]),
        "ck_fanout_plan": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]),
        "ck_tailcall_plan": (C.c_int, [vp, C.c_uint64, C.c_uint64]),
        "ck_exchange_plan": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i64p, i64p,
                                       C.POINTER(C.c_uint32)]),
        "ck_reply_plan": (C.c_int, [vp, C.c_uint32]),
        "ck_sync": (C.c_int, [vp]),
        "ck_launch_count": (C.c_uint64, [vp]),
        "ck_out_size": (C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "ck_fetch_columns": (C.c_int, [vp, u32p]),
        "ck_fetch_output": (C.c_int, [vp, u8p, C.c_uint64, i64p, u32p, vp]),
        "ck_fetch_cols": (C.c_int, [vp, u32p, C.c_uint32, u32p]),
        "ck_fetch_cols_async": (C.c_int, [vp, u32p, C.c_uint32, u32p]),
        "ck_fetch_output_async": (C.c_int, [vp, u8p, C.c_uint64, i64p, u32p, vp]),
        "ck_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(vp)]),
        "ck_host_free": (None, [vp]),
        "ck_canon_stats": (C.c_int, [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
        "ck_comm_create": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, u8p]),
        "ck_comm_connect": (C.c_int, [vp, u8p]),
        "ck_exchange_send": (C.c_int, [vp, C.c_uint64]),
        "ck_recv_info": (C.c_int, [vp, C.POINTER(vp), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
        "ck_fetch_received": (C.c_int, [vp, C.c_uint32, vp, u8p, u8p, C.c_uint64]),
        "ck_peek_received": (C.c_int, [vp, vp]),
        "ck_fetch_received_async": (C.c_int, [vp, C.c_uint32, C.c_uint64, C.c_uint64, u8p, u8p]),
        "ck_set_option": (C.c_int, [vp, C.c_uint32, C.c_uint64]),
        "ck_group_publishes": (C.c_int, [vp]),
        "ck_fetch_groups": (C.c_int, [vp, u32p, u32p, C.c_int]),
        "ck_submit_recordbatch": (C.c_int, [vp, u8p, C.c_uint64, C.POINTER(C.c_uint32)]),
        "ck_fetch_rb_index": (C.c_int, [vp, i64p, u32p, i64p, i32p, i64p, i32p, u32p]),
        "ck_fetch_rb_decompressed": (C.c_int, [vp, u8p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "ck_encode_recordbatch": (C.c_int, [vp, u32p, C.c_uint32, C.c_int64, C.c_int64, u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
        "ck_encode_recordbatches": (C.c_int, [vp, u32p, C.c_uint32, u32p, C.c_uint32, i64p, C.c_int64, C.c_uint32, C.c_uint32,
                                              C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
        "ck_fetch_recordbatches": (C.c_int, [vp, u8p, C.c_uint64, vp, u32p]),
        "ck_gate_create": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint64]),
        "ck_gate_register": (C.c_int, [vp, C.c_uint32]),
        "ck_gate_arrive": (C.c_int, [vp, C.c_uint64]),
        "ck_gate_stats": (C.c_int, [vp, vp]),
        "ck_gate_reset": (C.c_int, [vp]),
        "ck_fetch_overlay": (C.c_int, [vp, u8p, C.c_uint64, i64p, u32p, C.POINTER(C.c_uint64)]),
        "ck_fetch_topic_hist": (C.c_int, [vp, u32p, C.c_uint32]),
        "ck_stream": (vp, [vp]),
        "ck_device_buffers": (C.c_int, [vp] + [C.POINTER(vp)] * 5),
        "ck_device_buffers2": (C.c_int, [vp] + [C.POINTER(vp)] * 3),
        "ck_gather_spans": (C.c_int, [vp, u8p, i64p, i64p, C.c_uint32, u8p, i64p]),
        "ck_profile": (C.c_int, [vp, C.c_int]),
        "ck_profile_read": (C.c_int, [vp, vp, vp, C.c_int]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)      # AttributeError here = the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def ptr(a) -> int | None:
    """address of a numpy array / torch tensor / None"""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(type(a))
