"""ctypes binding of include/b200comms.h (libb200comms.so).

This is the binding a test or bench process uses; a Pothos process goes through the C++
block layer (pothoscomms_b200/blocks/) instead.  There is NO fallback: if the CUDA library
is missing this raises, and every compute entry point returns an error without a B200.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200comms.so")

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOMEM = 0, -1, -2, -3, -4

F32, CF32, F64, CF64, I8, CI8, I16, CI16, I32, CI32, I64, CI64 = range(12)
TAPS_REAL, TAPS_COMPLEX = 0, 1

DTYPE_CODES = {
    "float32": F32, "complex_float32": CF32, "float64": F64, "complex_float64": CF64,
    "int8": I8, "complex_int8": CI8, "int16": I16, "complex_int16": CI16,
    "int32": I32, "complex_int32": CI32, "int64": I64, "complex_int64": CI64,
}

# every symbol include/b200comms.h declares: (restype, argtypes)
_sz, _vp, _i = ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int
_psz, _pvp, _pi = ctypes.POINTER(_sz), ctypes.POINTER(_vp), ctypes.POINTER(_i)
SYMBOLS = {
    "b200c_last_error": (ctypes.c_char_p, []),
    "b200c_abi_version": (_i, []),
    "b200c_device_count": (_i, [_pi]),
    "b200c_dtype_size": (_sz, [_i]),
    "b200c_scale": (_i, [_i, ctypes.c_double, _vp, _vp, _sz, _i, _vp]),
    "b200c_rotate": (_i, [_i, ctypes.c_double, _vp, _vp, _sz, _i, _vp]),
    "b200c_probe": (_i, [_i, _i, _vp, _sz, ctypes.POINTER(ctypes.c_double), _i, _vp]),
    "b200c_table_source": (_i, [_i, _vp, _sz, ctypes.c_uint64, ctypes.c_uint64, _vp, _sz, _i, _vp]),
    "b200c_fir_create": (_i, [_pvp, _i, _i, _i]),
    "b200c_fir_destroy": (_i, [_vp]),
    "b200c_fir_set_taps": (_i, [_vp, _vp, _sz]),
    "b200c_fir_set_rates": (_i, [_vp, _sz, _sz]),
    "b200c_fir_info": (_i, [_vp, _psz, _psz, _psz, _psz]),
    "b200c_fir_kernel": (ctypes.c_char_p, [_vp]),
    "b200c_fir_plan": (_i, [_vp, _sz, _sz, _i, _psz, _psz]),
    "b200c_fir_run": (_i, [_vp, _vp, _sz, _vp, _sz, _i, _psz, _psz, _vp]),
    "b200c_fir_run_host": (_i, [_vp, _vp, _sz, _vp, _sz, _i, _psz, _psz]),
    "b200c_fir_bank_create": (_i, [_pvp, _i, _i, _sz, _i]),
    "b200c_fir_bank_destroy": (_i, [_vp]),
    "b200c_fir_bank_set_taps": (_i, [_vp, _sz, _vp, _sz]),
    "b200c_fir_bank_set_rates": (_i, [_vp, _sz, _sz]),
    "b200c_fir_bank_info": (_i, [_vp, _psz, _psz, _psz]),
    "b200c_fir_bank_run": (_i, [_vp, _vp, _sz, _sz, _vp, _sz, _sz, _i, _psz, _psz, _vp]),
    "b200c_chan_create": (_i, [_pvp, _i, _sz, _sz, _i]),
    "b200c_chan_destroy": (_i, [_vp]),
    "b200c_chan_set_taps": (_i, [_vp, _vp, _sz]),
    "b200c_chan_info": (_i, [_vp, _psz, _psz, _psz, _psz]),
    # stream_index is a uint64: a default int conversion would cut it to 32 bits
    "b200c_chan_run": (_i, [_vp, _vp, _sz, ctypes.c_uint64, _vp, _sz, _sz, _psz, _psz, _vp]),
    "b200c_rchan_create": (_i, [_pvp, _i, _sz, _sz, _i]),
    "b200c_rchan_destroy": (_i, [_vp]),
    "b200c_rchan_set_taps": (_i, [_vp, _vp, _sz]),
    "b200c_rchan_info": (_i, [_vp, _psz, _psz, _psz, _psz, _psz]),
    # stream_index is a uint64, as for b200c_chan_run
    "b200c_rchan_run": (_i, [_vp, _vp, _sz, ctypes.c_uint64, _vp, _sz, _sz, _psz, _psz, _vp]),
    "b200c_synth_create": (_i, [_pvp, _i, _sz, _sz, _i]),
    "b200c_synth_destroy": (_i, [_vp]),
    "b200c_synth_set_taps": (_i, [_vp, _vp, _sz]),
    "b200c_synth_info": (_i, [_vp, _psz, _psz, _psz, _psz]),
    # stream_index is a uint64, as for b200c_chan_run
    "b200c_synth_run": (_i, [_vp, _vp, _sz, _sz, ctypes.c_uint64, _vp, _sz, _psz, _psz, _vp]),
    "b200c_fft_create": (_i, [_pvp, _i, _sz, _i, _i]),
    "b200c_fft_destroy": (_i, [_vp]),
    "b200c_fft_info": (_i, [_vp, _psz, _pi]),
    "b200c_fft_run": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "b200c_fft_run_host": (_i, [_vp, _vp, _vp, _sz]),
    "b200c_ring_create": (_i, [_pvp, _sz, _i]),
    "b200c_ring_destroy": (_i, [_vp]),
    "b200c_ring_base": (_vp, [_vp]),
    "b200c_ring_bytes": (_sz, [_vp]),
    "b200c_dev_alloc": (_i, [_pvp, _sz, _i]),
    "b200c_dev_free": (_i, [_vp, _i]),
    "b200c_host_alloc_pinned": (_i, [_pvp, _sz]),
    "b200c_host_free_pinned": (_i, [_vp]),
    "b200c_copy_h2d": (_i, [_vp, _vp, _sz, _i, _vp]),
    "b200c_copy_d2h": (_i, [_vp, _vp, _sz, _i, _vp]),
    "b200c_copy_d2d": (_i, [_vp, _vp, _sz, _i, _vp]),
    "b200c_memset": (_i, [_vp, _i, _sz, _i, _vp]),
    "b200c_stream_sync": (_i, [_i, _vp]),
    # multi-GPU halo (b200c_peer_mem / b200c_peer_event are 128-byte PODs passed as raw buffers)
    "b200c_peer_export": (_i, [_vp, _sz, _i, _vp]),
    "b200c_peer_open": (_i, [_vp, _i, _pvp, _pvp]),
    "b200c_peer_close": (_i, [_vp]),
    "b200c_peer_event_create": (_i, [_pvp, _i, _vp]),
    "b200c_peer_event_open": (_i, [_vp, _i, _pvp]),
    "b200c_peer_event_record": (_i, [_vp, _i, _vp]),
    "b200c_peer_event_wait": (_i, [_vp, _i, _vp]),
    "b200c_peer_event_destroy": (_i, [_vp, _i]),
    "b200c_halo_exchange": (_i, [_vp, _vp, _sz, _i, _vp]),
}
PEER_RECORD_BYTES = 128   # sizeof(b200c_peer_mem) == sizeof(b200c_peer_event)


class B200CommsError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"[b200c {code}] {text}")
        self.code = code


class InvalidArgumentError(B200CommsError, ValueError):
    """What the block layer raises as Pothos::InvalidArgumentException."""


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the B200 path)")
        _lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def last_error() -> str:
    return lib().b200c_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc == OK:
        return
    text = last_error()
    if rc in (ERR_INVALID, ERR_UNSUPPORTED):
        raise InvalidArgumentError(rc, text)
    raise B200CommsError(rc, text)
