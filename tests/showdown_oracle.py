"""ctypes front-end of tests/showdown_oracle.c: the literal CPU enumeration that libnpk's exact showdown equity is checked
against.  Compiled with the C compiler into a temporary directory on first use (the repository tree may be read-only); hands
are scored with the oracle's oracle_rank7_fast."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
_rank7 = None


def lib():
    global _lib, _rank7
    if _lib is None:
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if not cc:
            raise RuntimeError("no C compiler for tests/showdown_oracle.c")
        tmp = tempfile.mkdtemp(prefix="npk_showdown_oracle_")
        try:
            out = os.path.join(tmp, "libshowdown_oracle.so")
            subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-Wall",
                                   os.path.join(HERE, "showdown_oracle.c"), "-o", out])
            L = ctypes.CDLL(out)                   # stays mapped after the file is gone
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        u8p = ctypes.POINTER(ctypes.c_uint8)
        L.showdown_equity.argtypes = [ctypes.c_void_p, u8p, ctypes.c_int, u8p, ctypes.c_int, ctypes.c_uint64, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_int64)]
        O = oracle.lib()
        O.oracle_fast_init()
        _rank7 = ctypes.cast(O.oracle_rank7_fast, ctypes.c_void_p)
        _lib = L
    return _lib


def showdown_equity(hands, board, dead=(), deal_mode="uniform"):
    """Exact showdown equity of known hands (every completion of the board): dict(win, tie, share, completions), one
    entry per hand; deal_mode "reference" leaves the highest unseen id out of the completions."""
    L = lib()
    h = np.ascontiguousarray([oracle.ids(x) for x in hands], dtype=np.uint8).reshape(-1)
    b = oracle.ids(board)
    mask = 0
    for c in oracle.ids(dead):
        mask |= 1 << int(c)
    P = len(hands)
    out = (ctypes.c_int64 * (3 * P + 1))()
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
    rc = L.showdown_equity(_rank7, p(h), P, p(b) if len(b) else None, len(b), mask, 1 if deal_mode == "reference" else 0, out)
    if rc:
        raise ValueError("showdown_equity oracle rc=%d" % rc)
    return {"win": list(out[:P]), "tie": list(out[P:2 * P]), "share": list(out[2 * P:3 * P]), "completions": out[3 * P]}
