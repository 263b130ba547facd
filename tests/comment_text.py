"""Generated comment text as (blob, offsets) arrays, for uploading millions of VARCHAR rows without a Python object per row
(DeviceTable.append takes that pair).  Cut from the oracle's text pool with one tg_comment_spans call per range; the same text
as oracle.comments(column, range(lo, hi))."""
import ctypes as C

import numpy as np


def comment_blob(oracle, column, lo, hi):
    """rows [lo, hi) of `column`: (blob uint8 array, offsets int64 array of hi - lo + 1), row r being
    blob[offsets[r - lo]:offsets[r - lo + 1]]"""
    L = oracle.lib()
    L.tg_text_pool.restype = C.c_void_p
    L.tg_comment_spans.restype = None
    L.tg_comment_spans.argtypes = [C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
    base = L.tg_text_pool()
    assert base, "text pool allocation failed"
    seed, avg = oracle.COMMENT_STREAMS[column]
    n = hi - lo
    off, ln = np.empty(n, np.int64), np.empty(n, np.int32)
    L.tg_comment_spans(seed, avg, lo, hi, off.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p))
    offsets = np.zeros(n + 1, np.int64)
    np.cumsum(ln, out=offsets[1:])
    if n == 0:
        return np.zeros(0, np.uint8), offsets
    width = int(ln.max())
    pool = np.ctypeslib.as_array((C.c_uint8 * (int(off.max()) + width)).from_address(base))
    win = np.lib.stride_tricks.sliding_window_view(pool, width)[off]          # every row's span, padded to the longest
    return win[np.arange(width) < ln[:, None]], offsets
