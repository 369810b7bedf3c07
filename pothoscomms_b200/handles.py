"""Thin Python owners of the C-ABI handles (FIR, FFT, device ring) for tests and bench.

Device buffers are torch CUDA tensors in the *raw* layout the ABI uses: shape [n, ncomp] of the
scalar type (ncomp = 2 for complex, interleaved re/im), so integer complex types need no
special casing.  torch is plumbing here (allocation + streams); all arithmetic happens in
libb200comms.so.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _abi

_NP_SCALAR = {0: np.float32, 1: np.float64, 2: np.int8, 3: np.int16, 4: np.int32, 5: np.int64}


def dtype_code(dtype) -> int:
    if isinstance(dtype, str):
        try:
            return _abi.DTYPE_CODES[dtype]
        except KeyError:
            raise _abi.InvalidArgumentError(_abi.ERR_UNSUPPORTED, f"unknown dtype {dtype!r}") from None
    return int(dtype)


def np_scalar(code: int):
    return _NP_SCALAR[code >> 1]


def ncomp(code: int) -> int:
    return 2 if code & 1 else 1


def torch_scalar(code: int):
    import torch
    return {0: torch.float32, 1: torch.float64, 2: torch.int8, 3: torch.int16, 4: torch.int32, 5: torch.int64}[code >> 1]


def _stream_ptr(stream, device):
    import torch
    if stream is None:
        stream = torch.cuda.current_stream(device)
    return ctypes.c_void_p(stream.cuda_stream)


def _taps_array(taps, complex_taps: bool) -> np.ndarray:
    if complex_taps:
        return np.ascontiguousarray(np.asarray(taps, dtype=np.complex128)).view(np.float64)
    arr = np.asarray(taps)
    if np.iscomplexobj(arr):
        raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "complex taps given to a REAL-taps filter")
    return np.ascontiguousarray(arr, dtype=np.float64)


class FirFilter:
    """Owner of a b200c_fir handle (the arithmetic state of one /comms/fir_filter block)."""

    def __init__(self, dtype, taps_type: str = "REAL", device: int = 0):
        self.dtype = dtype_code(dtype)
        if taps_type not in ("REAL", "COMPLEX"):
            raise _abi.InvalidArgumentError(_abi.ERR_UNSUPPORTED, f"FIRFilterFactory: unsupported tapsType {taps_type!r}")
        self.complex_taps = taps_type == "COMPLEX"
        self.device = device
        self._h = ctypes.c_void_p()
        _abi.check(_abi.lib().b200c_fir_create(ctypes.byref(self._h), self.dtype, int(self.complex_taps), device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_fir_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):   # interpreter shutdown: module globals are already gone
            pass

    __del__ = close

    def set_taps(self, taps):
        t = _taps_array(taps, self.complex_taps)
        n = t.size // (2 if self.complex_taps else 1)
        _abi.check(_abi.lib().b200c_fir_set_taps(self._h, t.ctypes.data, n))

    def set_rates(self, decim: int, interp: int):
        if decim < 0 or interp < 0:
            raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "negative rate")
        _abi.check(_abi.lib().b200c_fir_set_rates(self._h, decim, interp))

    def info(self):
        K, req, M, L = (ctypes.c_size_t() for _ in range(4))
        _abi.check(_abi.lib().b200c_fir_info(self._h, ctypes.byref(K), ctypes.byref(req), ctypes.byref(M), ctypes.byref(L)))
        return K.value, req.value, M.value, L.value

    @property
    def kernel(self) -> str:
        return _abi.lib().b200c_fir_kernel(self._h).decode()

    @property
    def K(self) -> int:
        return self.info()[0]

    @property
    def input_require(self) -> int:
        return self.info()[1]

    def plan(self, in_elems: int, out_capacity: int, zero_tail: bool = False):
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_fir_plan(self._h, in_elems, out_capacity, int(zero_tail), ctypes.byref(c), ctypes.byref(p)))
        return c.value, p.value

    def default_capacity(self, in_elems: int, zero_tail: bool = False) -> int:
        K, _, M, L = self.info()
        return ((in_elems + (K - 1 if zero_tail else 0)) // M + 1) * L

    def run(self, d_in, out=None, out_capacity: int | None = None, zero_tail: bool = False, stream=None):
        """d_in: CUDA tensor [n, ncomp] (K-1 history elements first).  Returns (out[:produced], consumed, produced)."""
        import torch
        nc = ncomp(self.dtype)
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dtype == torch_scalar(self.dtype)
        n_in = d_in.numel() // nc
        if out_capacity is None:
            out_capacity = out.numel() // nc if out is not None else self.default_capacity(n_in, zero_tail)
        if out is None:
            out = torch.empty((max(out_capacity, 1), nc), dtype=d_in.dtype, device=d_in.device)
        assert out.is_cuda and out.is_contiguous() and out.numel() // nc >= out_capacity
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_fir_run(self._h, ctypes.c_void_p(d_in.data_ptr()), n_in, ctypes.c_void_p(out.data_ptr()),
                                            out_capacity, int(zero_tail), ctypes.byref(c), ctypes.byref(p),
                                            _stream_ptr(stream, d_in.device)))
        return out[: p.value], c.value, p.value

    def run_host(self, x_raw: np.ndarray, out: np.ndarray | None = None, out_capacity: int | None = None,
                 zero_tail: bool = False):
        """Host-buffer entry point (numpy or pinned memory viewed as numpy)."""
        nc = ncomp(self.dtype)
        x_raw = np.ascontiguousarray(x_raw, dtype=np_scalar(self.dtype)).reshape(-1, nc)
        n_in = x_raw.shape[0]
        if out_capacity is None:
            out_capacity = out.size // nc if out is not None else self.default_capacity(n_in, zero_tail)
        if out is None:
            out = np.empty((max(out_capacity, 1), nc), dtype=x_raw.dtype)
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_fir_run_host(self._h, x_raw.ctypes.data, n_in, out.ctypes.data, out_capacity,
                                                 int(zero_tail), ctypes.byref(c), ctypes.byref(p)))
        return out.reshape(-1, nc)[: p.value], c.value, p.value


class FirFilterBank:
    """Owner of a b200c_fir_bank handle: `nchan` FIR filter states run by one call (channeliser)."""

    def __init__(self, dtype, taps_type: str = "REAL", nchan: int = 1, device: int = 0):
        self.dtype = dtype_code(dtype)
        if taps_type not in ("REAL", "COMPLEX"):
            raise _abi.InvalidArgumentError(_abi.ERR_UNSUPPORTED, f"FIRFilterFactory: unsupported tapsType {taps_type!r}")
        self.complex_taps = taps_type == "COMPLEX"
        self.nchan = int(nchan)
        self.device = device
        self._h = ctypes.c_void_p()
        _abi.check(_abi.lib().b200c_fir_bank_create(ctypes.byref(self._h), self.dtype, int(self.complex_taps), self.nchan, device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_fir_bank_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close

    def set_taps(self, chan: int, taps):
        t = _taps_array(taps, self.complex_taps)
        n = t.size // (2 if self.complex_taps else 1)
        _abi.check(_abi.lib().b200c_fir_bank_set_taps(self._h, chan, t.ctypes.data, n))

    def set_rates(self, decim: int, interp: int):
        _abi.check(_abi.lib().b200c_fir_bank_set_rates(self._h, decim, interp))

    def info(self):
        n, K, req = (ctypes.c_size_t() for _ in range(3))
        _abi.check(_abi.lib().b200c_fir_bank_info(self._h, ctypes.byref(n), ctypes.byref(K), ctypes.byref(req)))
        return n.value, K.value, req.value

    def run(self, d_in, out, zero_tail: bool = False, stream=None):
        """d_in: CUDA tensor [nchan, n_in, ncomp]; out: CUDA tensor [nchan, capacity, ncomp].
        Returns (consumed, produced) per channel."""
        import torch
        nc = ncomp(self.dtype)
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dtype == torch_scalar(self.dtype) and d_in.shape[0] == self.nchan
        assert out.is_cuda and out.is_contiguous() and out.shape[0] == self.nchan
        n_in, cap = d_in.shape[1], out.shape[1]
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_fir_bank_run(self._h, ctypes.c_void_p(d_in.data_ptr()), n_in, n_in, ctypes.c_void_p(out.data_ptr()),
                                                 cap, cap, int(zero_tail), ctypes.byref(c), ctypes.byref(p),
                                                 _stream_ptr(stream, d_in.device)))
        return c.value, p.value


class Channelizer:
    """Owner of a b200c_chan handle: one complex float32 stream into `nchan` baseband channels (polyphase
    filter bank), decimated by `decim`.  Channel c is /comms/fir_filter with the real prototype taps applied to
    the stream mixed down by c/nchan cycles per sample (include/b200comms.h has the exact definition)."""

    def __init__(self, dtype, nchan: int, decim: int, device: int = 0):
        self.dtype = dtype_code(dtype)
        self.nchan = int(nchan)
        self.decim = int(decim)
        self.device = device
        self._h = ctypes.c_void_p()
        if self.nchan < 0 or self.decim < 0:
            raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "negative channel count or decimation")
        _abi.check(_abi.lib().b200c_chan_create(ctypes.byref(self._h), self.dtype, self.nchan, self.decim, device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_chan_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close

    def set_taps(self, taps):
        t = _taps_array(taps, False)
        _abi.check(_abi.lib().b200c_chan_set_taps(self._h, t.ctypes.data, t.size))

    def info(self):
        """(nchan, decim, ntaps, input_require)"""
        n, d, k, req = (ctypes.c_size_t() for _ in range(4))
        _abi.check(_abi.lib().b200c_chan_info(self._h, ctypes.byref(n), ctypes.byref(d), ctypes.byref(k), ctypes.byref(req)))
        return n.value, d.value, k.value, req.value

    def run(self, d_in, out, stream_index: int = 0, out_capacity: int | None = None, stream=None):
        """d_in: CUDA tensor [n, 2] float32 (ntaps-1 history samples first); out: CUDA tensor [nchan, capacity, 2]
        float32, frame t of channel c lands in out[c, t].  stream_index: absolute stream index of d_in[0].
        Returns (consumed, produced)."""
        import torch
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dtype == torch.float32
        assert out.is_cuda and out.is_contiguous() and out.dtype == torch.float32 and out.dim() == 3 and out.shape[0] == self.nchan
        stride = out.shape[1]
        cap = stride if out_capacity is None else int(out_capacity)
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_chan_run(self._h, ctypes.c_void_p(d_in.data_ptr()), d_in.numel() // 2,
                                             int(stream_index) & (2**64 - 1), ctypes.c_void_p(out.data_ptr()), stride, cap,
                                             ctypes.byref(c), ctypes.byref(p), _stream_ptr(stream, d_in.device)))
        return c.value, p.value


class RealChannelizer:
    """Owner of a b200c_rchan handle: one real float32 or int16 stream into M/2 + 1 baseband channels (polyphase
    filter bank with M branches), decimated by `decim`.  Channel c is the Channelizer's channel c of the stream
    taken as complex; the channels above M/2 are their conjugate mirrors and are not produced (include/b200comms.h
    has the exact definition)."""

    def __init__(self, dtype, m: int, decim: int, device: int = 0):
        self.dtype = dtype_code(dtype)
        self.m = int(m)
        self.nchan = self.m // 2 + 1
        self.decim = int(decim)
        self.device = device
        self._h = ctypes.c_void_p()
        if self.m < 0 or self.decim < 0:
            raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "negative branch count or decimation")
        _abi.check(_abi.lib().b200c_rchan_create(ctypes.byref(self._h), self.dtype, self.m, self.decim, device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_rchan_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close

    def set_taps(self, taps):
        t = _taps_array(taps, False)
        _abi.check(_abi.lib().b200c_rchan_set_taps(self._h, t.ctypes.data, t.size))

    def info(self):
        """(m, nchan, decim, ntaps, input_require), nchan = m/2 + 1"""
        m, n, d, k, req = (ctypes.c_size_t() for _ in range(5))
        _abi.check(_abi.lib().b200c_rchan_info(self._h, ctypes.byref(m), ctypes.byref(n), ctypes.byref(d), ctypes.byref(k),
                                               ctypes.byref(req)))
        return m.value, n.value, d.value, k.value, req.value

    def run(self, d_in, out, stream_index: int = 0, out_capacity: int | None = None, stream=None):
        """d_in: contiguous 1-D CUDA tensor of float32 or int16 (the handle's dtype; ntaps-1 history samples first);
        out: CUDA tensor [m/2 + 1, capacity, 2] float32, frame t of channel c lands in out[c, t].  stream_index:
        absolute stream index of d_in[0].  Returns (consumed, produced)."""
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dim() == 1 and d_in.dtype == torch_scalar(self.dtype)
        assert out.is_cuda and out.is_contiguous() and out.dim() == 3 and out.shape[0] == self.nchan
        assert out.dtype == torch_scalar(_abi.F32)
        stride = out.shape[1]
        cap = stride if out_capacity is None else int(out_capacity)
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_rchan_run(self._h, ctypes.c_void_p(d_in.data_ptr()), d_in.numel(),
                                              int(stream_index) & (2**64 - 1), ctypes.c_void_p(out.data_ptr()), stride, cap,
                                              ctypes.byref(c), ctypes.byref(p), _stream_ptr(stream, d_in.device)))
        return c.value, p.value


class Synthesizer:
    """Owner of a b200c_synth handle: `nchan` baseband channels, interpolated by `interp`, back into one complex
    float32 stream (polyphase synthesis filter bank, the transpose of Channelizer).  Channel c is /comms/fir_filter
    with the real prototype taps and interpolation `interp`, mixed up by +c/nchan cycles per sample, and the channels
    are summed (include/b200comms.h has the exact definition)."""

    def __init__(self, dtype, nchan: int, interp: int, device: int = 0):
        self.dtype = dtype_code(dtype)
        self.nchan = int(nchan)
        self.interp = int(interp)
        self.device = device
        self._h = ctypes.c_void_p()
        if self.nchan < 0 or self.interp < 0:
            raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "negative channel count or interpolation")
        _abi.check(_abi.lib().b200c_synth_create(ctypes.byref(self._h), self.dtype, self.nchan, self.interp, device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_synth_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close

    def set_taps(self, taps):
        t = _taps_array(taps, False)
        _abi.check(_abi.lib().b200c_synth_set_taps(self._h, t.ctypes.data, t.size))

    def info(self):
        """(nchan, interp, ntaps, input_require), input_require = ceil(ntaps / interp) frames"""
        n, d, k, req = (ctypes.c_size_t() for _ in range(4))
        _abi.check(_abi.lib().b200c_synth_info(self._h, ctypes.byref(n), ctypes.byref(d), ctypes.byref(k), ctypes.byref(req)))
        return n.value, d.value, k.value, req.value

    def run(self, d_in, out, stream_index: int = 0, in_frames: int | None = None, out_capacity: int | None = None,
            stream=None):
        """d_in: CUDA tensor [nchan, stride, 2] float32, frame i of channel c in d_in[c, i] (the Channelizer's output
        layout; the first ceil(ntaps/interp)-1 frames are history); out: CUDA tensor [n, 2] float32.
        stream_index: absolute stream index of out[0].  Returns (consumed frames per channel, produced samples)."""
        import torch
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dtype == torch.float32
        assert d_in.dim() == 3 and d_in.shape[0] == self.nchan
        assert out.is_cuda and out.is_contiguous() and out.dtype == torch.float32
        stride = d_in.shape[1]
        frames = stride if in_frames is None else int(in_frames)
        cap = out.numel() // 2 if out_capacity is None else int(out_capacity)
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_synth_run(self._h, ctypes.c_void_p(d_in.data_ptr()), stride, frames,
                                              int(stream_index) & (2**64 - 1), ctypes.c_void_p(out.data_ptr()), cap,
                                              ctypes.byref(c), ctypes.byref(p), _stream_ptr(stream, d_in.device)))
        return c.value, p.value


class RealSynthesizer:
    """Owner of a b200c_rsynth handle: the M/2 + 1 baseband channels of a RealChannelizer (polyphase filter bank with
    M branches), interpolated by `interp`, back into one real float32 or int16 stream.  The output is the real part of
    the Synthesizer's at M channels with rows M - c taken as conj(row c); int16 output is rounded to nearest and
    saturated (include/b200comms.h has the exact definition)."""

    def __init__(self, dtype, m: int, interp: int, device: int = 0):
        self.dtype = dtype_code(dtype)
        self.m = int(m)
        self.nchan = self.m // 2 + 1
        self.interp = int(interp)
        self.device = device
        self._h = ctypes.c_void_p()
        if self.m < 0 or self.interp < 0:
            raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "negative branch count or interpolation")
        _abi.check(_abi.lib().b200c_rsynth_create(ctypes.byref(self._h), self.dtype, self.m, self.interp, device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_rsynth_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close

    def set_taps(self, taps):
        t = _taps_array(taps, False)
        _abi.check(_abi.lib().b200c_rsynth_set_taps(self._h, t.ctypes.data, t.size))

    def info(self):
        """(m, nchan, interp, ntaps, input_require), nchan = m/2 + 1, input_require = ceil(ntaps / interp) frames"""
        m, n, d, k, req = (ctypes.c_size_t() for _ in range(5))
        _abi.check(_abi.lib().b200c_rsynth_info(self._h, ctypes.byref(m), ctypes.byref(n), ctypes.byref(d), ctypes.byref(k),
                                                ctypes.byref(req)))
        return m.value, n.value, d.value, k.value, req.value

    def run(self, d_in, out, stream_index: int = 0, in_frames: int | None = None, out_capacity: int | None = None,
            stream=None):
        """d_in: CUDA tensor [m/2 + 1, stride, 2] float32, frame i of row c in d_in[c, i] (the RealChannelizer's output
        layout; the first ceil(ntaps/interp)-1 frames are history); out: contiguous 1-D CUDA tensor of float32 or int16
        (the handle's dtype), which may start at any element.  stream_index: absolute stream index of out[0].
        Returns (consumed frames per row, produced samples)."""
        import torch
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dtype == torch.float32
        assert d_in.dim() == 3 and d_in.shape[0] == self.nchan and d_in.shape[2] == 2
        assert out.is_cuda and out.is_contiguous() and out.dim() == 1 and out.dtype == torch_scalar(self.dtype)
        stride = d_in.shape[1]
        frames = stride if in_frames is None else int(in_frames)
        cap = out.numel() if out_capacity is None else int(out_capacity)
        c, p = ctypes.c_size_t(), ctypes.c_size_t()
        _abi.check(_abi.lib().b200c_rsynth_run(self._h, ctypes.c_void_p(d_in.data_ptr()), stride, frames,
                                               int(stream_index) & (2**64 - 1), ctypes.c_void_p(out.data_ptr()), cap,
                                               ctypes.byref(c), ctypes.byref(p), _stream_ptr(stream, d_in.device)))
        return c.value, p.value


class Fft:
    """Owner of a b200c_fft handle (the FFTAux of one /comms/fft block)."""

    def __init__(self, dtype, num_bins: int, inverse: bool = False, device: int = 0):
        self.dtype = dtype_code(dtype)
        self.num_bins = int(num_bins)
        self.inverse = bool(inverse)
        self.device = device
        self._h = ctypes.c_void_p()
        if self.num_bins < 0:
            raise _abi.InvalidArgumentError(_abi.ERR_INVALID, "negative numBins")
        _abi.check(_abi.lib().b200c_fft_create(ctypes.byref(self._h), self.dtype, self.num_bins, int(self.inverse), device))

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_fft_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close

    def run(self, d_in, out=None, stream=None):
        import torch
        assert d_in.is_cuda and d_in.is_contiguous() and d_in.dtype == torch_scalar(self.dtype)
        batch = (d_in.numel() // 2) // self.num_bins
        if out is None:
            out = torch.empty((batch * self.num_bins, 2), dtype=d_in.dtype, device=d_in.device)
        assert out.is_cuda and out.is_contiguous() and out.numel() >= batch * self.num_bins * 2
        _abi.check(_abi.lib().b200c_fft_run(self._h, ctypes.c_void_p(d_in.data_ptr()), ctypes.c_void_p(out.data_ptr()), batch,
                                            _stream_ptr(stream, d_in.device)))
        return out

    def run_host(self, x_raw: np.ndarray, out: np.ndarray | None = None):
        x_raw = np.ascontiguousarray(x_raw, dtype=np_scalar(self.dtype)).reshape(-1, 2)
        batch = x_raw.shape[0] // self.num_bins
        if out is None:
            out = np.empty((batch * self.num_bins, 2), dtype=x_raw.dtype)
        _abi.check(_abi.lib().b200c_fft_run_host(self._h, x_raw.ctypes.data, out.ctypes.data, batch))
        return out


class DeviceRing:
    """VMM double-mapped HBM ring: base[off : off+len] is contiguous for any off < bytes."""

    def __init__(self, min_bytes: int, device: int = 0):
        self.device = device
        self._h = ctypes.c_void_p()
        _abi.check(_abi.lib().b200c_ring_create(ctypes.byref(self._h), min_bytes, device))
        self.base = _abi.lib().b200c_ring_base(self._h)
        self.bytes = _abi.lib().b200c_ring_bytes(self._h)

    def close(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                _abi.lib().b200c_ring_destroy(self._h)
                self._h = ctypes.c_void_p()
        except (TypeError, AttributeError):
            pass

    __del__ = close


# ------------------------------------------------------- HBM-resident neighbours (SURVEY 8f) ---
def _raw_cuda(x, code):
    assert x.is_cuda and x.is_contiguous() and x.dtype == torch_scalar(code)
    return x.numel() // ncomp(code)


def scale(dtype, factor: float, d_in, out=None, stream=None):
    """/comms/scale on a CUDA tensor of raw scalars ([n, ncomp]); returns the output tensor."""
    import torch
    code = dtype_code(dtype)
    n = _raw_cuda(d_in, code)
    if out is None:
        out = torch.empty_like(d_in)
    _abi.check(_abi.lib().b200c_scale(code, float(factor), ctypes.c_void_p(d_in.data_ptr()), ctypes.c_void_p(out.data_ptr()), n,
                                      d_in.device.index or 0, _stream_ptr(stream, d_in.device)))
    return out


def rotate(dtype, phase: float, d_in, out=None, stream=None):
    """/comms/rotate on a CUDA tensor [n, 2] of a complex type."""
    import torch
    code = dtype_code(dtype)
    if not code & 1:
        raise _abi.InvalidArgumentError(_abi.ERR_UNSUPPORTED, "rotateFactory(): unsupported type")
    n = _raw_cuda(d_in, code)
    if out is None:
        out = torch.empty_like(d_in)
    _abi.check(_abi.lib().b200c_rotate(code, float(phase), ctypes.c_void_p(d_in.data_ptr()), ctypes.c_void_p(out.data_ptr()), n,
                                       d_in.device.index or 0, _stream_ptr(stream, d_in.device)))
    return out


PROBE_MODES = {"VALUE": 0, "RMS": 1, "MEAN": 2}


def probe(dtype, mode: str, d_in, stream=None) -> complex:
    """/comms/signal_probe over the whole tensor (one window); synchronous."""
    code = dtype_code(dtype)
    n = _raw_cuda(d_in, code)
    v = (ctypes.c_double * 2)()
    _abi.check(_abi.lib().b200c_probe(code, PROBE_MODES[mode], ctypes.c_void_p(d_in.data_ptr()), n, v, d_in.device.index or 0,
                                      _stream_ptr(stream, d_in.device)))
    return complex(v[0], v[1])


def table_source(dtype, d_table, index: int, step: int, elems: int, out=None, stream=None):
    """The work() loop of /comms/waveform_source / /comms/noise_source: out[i] = table[(index + i*step) & mask]
    from a CUDA table tensor of raw scalars ([entries, ncomp], entries a power of two)."""
    import torch
    code = dtype_code(dtype)
    entries = _raw_cuda(d_table, code)
    if out is None:
        out = torch.empty((elems, ncomp(code)), dtype=d_table.dtype, device=d_table.device)
    _abi.check(_abi.lib().b200c_table_source(code, ctypes.c_void_p(d_table.data_ptr()), entries, index & (2**64 - 1),
                                             step & (2**64 - 1), ctypes.c_void_p(out.data_ptr()), elems,
                                             d_table.device.index or 0, _stream_ptr(stream, d_table.device)))
    return out
