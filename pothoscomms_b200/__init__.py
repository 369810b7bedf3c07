"""pothoscomms_b200 -- B200-native /comms/fir_filter + /comms/fft (PothosComms hot path).

Layout:
  csrc/        hand-written sm_100a CUDA kernels + the extern "C" ABI (libb200comms.so)
  blocks/      C++ block layer mirroring the Pothos plugin surface (registry paths, calls)
  _abi.py      ctypes binding of include/b200comms.h
  handles.py   Python owners of the ABI handles for tests/bench: FirFilter, FirFilterBank, Channelizer
               (complex stream into M channels), RealChannelizer (real float32 / int16 stream into M/2 + 1
               channels), Synthesizer (M channels back into one stream), Fft, DeviceRing
  workloads.py synthetic taps + tone/noise input of BASELINE.json's configs

Importing this package loads libb200comms.so; a missing library is an ImportError (there
is no CPU fallback path anywhere in the package).
"""
from . import _abi
from ._abi import B200CommsError, InvalidArgumentError

_abi.lib()  # fail loudly at import time if the CUDA library is not built

from .handles import Channelizer, DeviceRing, Fft, FirFilter, FirFilterBank, RealChannelizer, Synthesizer  # noqa: E402

__all__ = ["FirFilter", "FirFilterBank", "Channelizer", "RealChannelizer", "Synthesizer", "Fft", "DeviceRing", "B200CommsError", "InvalidArgumentError"]
