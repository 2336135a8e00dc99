"""ctypes binding of libnpk.so (include/npk.h).  The library is the product: if it (or a GPU) is missing every compute
entry point raises -- there is no CPU fallback."""
import ctypes
import os
import threading

from . import _build

_lock = threading.Lock()
_lib = None
_inited = set()

NPK_DEAL_UNIFORM = 0
NPK_DEAL_REFERENCE = 1
NPK_FLAG_VALIDATE = 1
ERRORS = {-1: "NPK_ERR_NOT_INITIALIZED", -2: "NPK_ERR_INVALID_ARGUMENT", -3: "NPK_ERR_CUDA", -4: "NPK_ERR_TABLES",
          -5: "NPK_ERR_INVALID_CARDS", -6: "NPK_ERR_RANGE"}


class NpkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (ERRORS.get(code, code), msg))
        self.code = code


def lib():
    """Load (building it first if the sources are newer) neuron_poker_b200/libnpk.so."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                path = os.environ.get("NPK_LIBRARY")            # an experimental build (tools/), never a fallback
                if not path:
                    path = _build.LIB
                    if not os.path.exists(path) or (_build.stale() and os.environ.get("NPK_NO_REBUILD") != "1"):
                        path = _build.build()
                L = ctypes.CDLL(path)
                vp, u8, u16, u32, u64, i64, i32 = (ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                    ctypes.c_void_p, ctypes.c_int64, ctypes.c_int)
                L.npk_last_error.restype = ctypes.c_char_p
                L.npk_init.argtypes = [i32]
                L.npk_set_device.argtypes = [i32]
                L.npk_get_tables.argtypes = [u16, ctypes.POINTER(ctypes.c_int64), u16, u16, u32, u16, u64]
                L.npk_host_rank7.argtypes = [u8, i64, u16]
                L.npk_equity_workspace_bytes.argtypes = [i64]
                L.npk_equity_workspace_bytes.restype = i64
                L.npk_equity_batch.argtypes = [u8, u8, u8, i64, i64, i32, i32, ctypes.c_uint64, i64, i64, i32,
                                               ctypes.c_uint32, u64, u64, u64, u64, vp, vp]
                L.npk_equity_batch_async.argtypes = [u8, u8, u8, i64, i64, ctypes.c_uint64, ctypes.c_uint64, i64, i64, i32,
                                                     u64, u64, u64, u64, vp, vp]
                L.npk_equity_batch_status.argtypes = [vp, vp, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]
                L.npk_equity_adaptive_workspace_bytes.argtypes = [i64]
                L.npk_equity_adaptive_workspace_bytes.restype = i64
                L.npk_equity_batch_adaptive.argtypes = [u8, u8, u8, i64, i64, i64, ctypes.c_double, ctypes.c_uint64,
                                                        ctypes.c_uint64, i64, i32, ctypes.c_uint32, u64, u64, u64, u64, u64,
                                                        vp, vp]
                L.npk_equity_host.argtypes = [u8, u8, u8, i64, i64, ctypes.c_uint64, i32, u64, u64, u64, u64]
                L.npk_equity_host_submit.argtypes = [u8, u8, u8, i64, i64, ctypes.c_uint64, i32, ctypes.c_uint32]
                L.npk_equity_host_submit.restype = i64
                L.npk_equity_host_wait.argtypes = [i64, u64, u64, u64, u64]
                L.npk_resident_start.argtypes = [i32, i32]
                L.npk_equity_one.argtypes = [ctypes.c_uint64, i32, i64, ctypes.c_uint64, i32, ctypes.c_uint32, u64]
                L.npk_equity_ranges_batch.argtypes = [u8, u8, u8, u8, i64, i64, u64, u64, ctypes.c_uint64, i64, i64, i32,
                                                      ctypes.c_uint32, u64, u64, u64, u64, vp, vp]
                L.npk_equity_ranges_host.argtypes = [u8, u8, u8, u8, i64, i64, u64, u64, ctypes.c_uint64, i32, u64, u64,
                                                     u64, u64]
                L.npk_equity_ranges_known_batch.argtypes = [u8, u8, u8, u8, u8, i32, i64, i64, u64, u64, ctypes.c_uint64, i64, i64,
                                                            i32, ctypes.c_uint32, u64, u64, u64, u64, vp, vp]
                L.npk_equity_ranges_batch_adaptive.argtypes = [u8, u8, u8, u8, u8, i32, i64, i64, i64, ctypes.c_double, u64,
                                                               u64, ctypes.c_uint64, i64, i32, ctypes.c_uint32, u64, u64, u64,
                                                               u64, u64, vp, vp]
                L.npk_equity_ranges_known_host.argtypes = [u8, u8, u8, u8, u8, i32, i64, i64, u64, u64, ctypes.c_uint64, i32,
                                                           u64, u64, u64, u64]
                L.npk_peer_create.argtypes = [i32, i32, i64, ctypes.POINTER(ctypes.c_void_p), vp]
                L.npk_peer_connect.argtypes = [vp, vp]
                L.npk_peer_destroy.argtypes = [vp]
                L.npk_peer_error.argtypes = [vp, ctypes.POINTER(ctypes.c_int)]
                L.npk_equity_batch_sharded.argtypes = [vp, u8, u8, u8, i64, i64, i32, i32, ctypes.c_uint64, i64, i32, u64, vp]
                L.npk_rank7_batch.argtypes = [u8, i64, u16, ctypes.c_uint32, vp]
                L.npk_rank7_colex.argtypes = [i64, i64, u16, vp]
                L.npk_enum_batch.argtypes = [u8, u8, u8, i64, u64, u64, u64, ctypes.c_uint32, vp]
                L.npk_showdown_batch.argtypes = [u8, u8, u8, i64, i32, vp, u8, u16, ctypes.c_uint32, vp]
                L.npk_showdown_equity_workspace_bytes.argtypes = [i64]
                L.npk_showdown_equity_workspace_bytes.restype = i64
                L.npk_showdown_equity_batch.argtypes = [u8, u8, u8, u64, i64, i32, i32, ctypes.c_uint32, u64, u64, u64, u64,
                                                        vp, vp]
                L.npk_checked_status.argtypes = [ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_uint32)]
                L.npk_int_peak.argtypes = [i32, i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)]
                L.npk_philox_debug.argtypes = [u32, ctypes.c_uint32, ctypes.c_uint32, i32, u32, vp]
                _lib = L
    return _lib


_fast = None


def fast():
    """The CPython binding of npk_equity_one (csrc/npk_pyfast.c), bound to the loaded libnpk.so; built on first use like the
    library itself.  A faster way into the same entry point, not another implementation."""
    global _fast
    if _fast is None:
        L = lib()
        with _lock:
            if _fast is None:
                import importlib.util
                path = _build.build_fast()
                spec = importlib.util.spec_from_file_location("_npkfast", path)
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                mod.bind(ctypes.cast(L.npk_equity_one, ctypes.c_void_p).value)
                _fast = mod
    return _fast


def check(rc):
    if rc < 0:
        raise NpkError(rc, lib().npk_last_error().decode())
    return rc


def init(device=0):
    """npk_init(device): build + upload the rank tables; raises NpkError when no B200 is usable."""
    L = lib()
    check(L.npk_init(int(device)))
    _inited.add(int(device))
    return L


_current = threading.local()


def ensure_init(device=0):
    """Initialise `device` on first use and make it current for this thread inside libnpk's CUDA runtime."""
    device = int(device)
    if device not in _inited:
        L = init(device)
    else:
        L = lib()
        check(L.npk_set_device(device))
    _current.device = device
    return L


def ensure_current(device):
    """ensure_init for callers that never switch devices behind libnpk's back (the one-query drop-in path): the
    cudaSetDevice round trip is skipped when this thread's last libnpk call already selected `device`."""
    if getattr(_current, "device", None) == device:
        return _lib
    return ensure_init(device)
