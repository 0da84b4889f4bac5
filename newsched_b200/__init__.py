"""newsched_b200 -- B200 (sm_100a) implementation of newsched's data-parallel block hot path.

The product is ``lib/libb200dsp.so`` (hand-written CUDA behind the C-ABI of
``include/b200dsp.h``) plus the C++17 block wrappers under ``include/gnuradio``.  This Python
package is a thin ctypes mirror of the same C-ABI used by the tests and by ``bench.py``;
PyTorch is only the plumbing for device memory and streams.

There is no CPU fallback: if the CUDA library is missing every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

__all__ = [
    "lib", "build", "B200Error", "copy", "multiply_const", "multiply", "add", "complex_to_mag", "FirFilter", "FFT",
    "PfbChannelizer", "Chain", "DeviceRing", "launch_count", "LIB_PATH", "IpcHandle", "ipc_export", "ipc_import",
    "ipc_close",
]

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200_LIB", os.path.join(_HERE, "lib", "libb200dsp.so"))
_lib = None

OUT_COMPLEX, OUT_MAG, OUT_MAG_SQUARED = 0, 1, 2
OP_COPY, OP_MULTIPLY_CONST_CC, OP_COMPLEX_TO_MAG, OP_FIR, OP_FFT, OP_PFB, OP_MULTIPLY_CONST_FF = 1, 2, 3, 4, 5, 6, 7


class B200Error(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile libb200dsp.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    if not verbose:
        cmd.append("-s")
    subprocess.check_call(cmd)
    return LIB_PATH


class _FirParams(C.Structure):
    _fields_ = [("taps", C.POINTER(C.c_float)), ("n_taps", C.c_int32), ("decimation", C.c_int32),
                ("is_complex", C.c_int32), ("fuse_multiply_const", C.c_int32), ("k_re", C.c_float),
                ("k_im", C.c_float), ("algorithm", C.c_int32)]


class _ResamplerParams(C.Structure):
    _fields_ = [("taps", C.POINTER(C.c_float)), ("n_taps", C.c_int32), ("interpolation", C.c_int32),
                ("decimation", C.c_int32), ("is_complex", C.c_int32)]


class _FftParams(C.Structure):
    _fields_ = [("n", C.c_int32), ("forward", C.c_int32), ("window", C.POINTER(C.c_float)),
                ("shift", C.c_int32), ("output", C.c_int32), ("fuse_pre_multiply_const", C.c_int32),
                ("k_re", C.c_float), ("k_im", C.c_float)]


class _PfbParams(C.Structure):
    _fields_ = [("taps", C.POINTER(C.c_float)), ("n_channels", C.c_int32),
                ("taps_per_channel", C.c_int32), ("channel_begin", C.c_int32),
                ("channel_count", C.c_int32), ("oversample", C.c_int32)]


class IpcHandle(C.Structure):
    """b200_ipc_handle: 88 plain bytes, shipped between processes over any host channel."""
    _fields_ = [("bytes", C.c_ubyte * 64), ("offset", C.c_uint64), ("size", C.c_uint64),
                ("device", C.c_int32), ("reserved", C.c_int32)]


class _ChainOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("handle", C.c_void_p), ("k_re", C.c_float), ("k_im", C.c_float)]


# name -> (restype, argtypes); this table is also what tests/test_cabi.py checks against
# include/b200dsp.h
_V, _I, _I64, _SZ, _F = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float
_PI64 = C.POINTER(C.c_int64)
SIGNATURES = {
    "b200_version": (_I, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_device_count": (_I, [C.POINTER(_I)]),
    "b200_set_device": (_I, [_I]),
    "b200_get_device": (_I, [C.POINTER(_I)]),
    "b200_device_sm_count": (_I, [C.POINTER(_I)]),
    "b200_device_synchronize": (_I, []),
    "b200_launch_count": (_I64, []),
    "b200_measure_fp32_tflops": (_I, [_I, C.POINTER(_F), C.POINTER(_F)]),
    "b200_measure_fp32x2_tflops": (_I, [_I, C.POINTER(_F), C.POINTER(_F)]),
    "b200_malloc": (_I, [C.POINTER(_V), _SZ]),
    "b200_free": (_I, [_V]),
    "b200_host_alloc": (_I, [C.POINTER(_V), _SZ]),
    "b200_host_free": (_I, [_V]),
    "b200_host_register": (_I, [_V, _SZ]),
    "b200_host_unregister": (_I, [_V]),
    "b200_memcpy_h2d": (_I, [_V, _V, _SZ, _V]),
    "b200_memcpy_d2h": (_I, [_V, _V, _SZ, _V]),
    "b200_memcpy_d2d": (_I, [_V, _V, _SZ, _V]),
    "b200_memset": (_I, [_V, _I, _SZ, _V]),
    "b200_stream_create": (_I, [C.POINTER(_V)]),
    "b200_stream_destroy": (_I, [_V]),
    "b200_stream_synchronize": (_I, [_V]),
    "b200_stream_activate": (_I, [_V]),
    "b200_stream_wait_event": (_I, [_V, _V]),
    "b200_event_create": (_I, [C.POINTER(_V), _I]),
    "b200_event_destroy": (_I, [_V]),
    "b200_event_record": (_I, [_V, _V]),
    "b200_event_synchronize": (_I, [_V]),
    "b200_event_query": (_I, [_V]),
    "b200_event_elapsed_ms": (_I, [_V, _V, C.POINTER(_F)]),
    "b200_enable_peer_access": (_I, [_I]),
    "b200_ipc_export": (_I, [_V, C.POINTER(IpcHandle)]),
    "b200_ipc_import": (_I, [C.POINTER(IpcHandle), C.POINTER(_V)]),
    "b200_ipc_close": (_I, [C.POINTER(IpcHandle), _V]),
    "b200_ring_create": (_I, [_SZ, C.POINTER(_V)]),
    "b200_ring_destroy": (_I, [_V]),
    "b200_ring_enable_peer": (_I, [_V, _I]),
    "b200_ring_base": (_V, [_V]),
    "b200_ring_size": (_SZ, [_V]),
    "b200_ring_granularity": (_SZ, []),
    "b200_copy": (_I, [_V, _V, _SZ, _V]),
    "b200_multiply_const_ff": (_I, [_V, _V, _F, _SZ, _V]),
    "b200_multiply_const_cc": (_I, [_V, _V, _F, _F, _SZ, _V]),
    "b200_multiply_const_ss": (_I, [_V, _V, C.c_int16, _SZ, _V]),
    "b200_multiply_const_ii": (_I, [_V, _V, C.c_int32, _SZ, _V]),
    "b200_multiply_ff": (_I, [_V, _V, _V, _SZ, _V]),
    "b200_multiply_cc": (_I, [_V, _V, _V, _SZ, _V]),
    "b200_add_ff": (_I, [_V, _V, _V, _SZ, _V]),
    "b200_add_cc": (_I, [_V, _V, _V, _SZ, _V]),
    "b200_complex_to_mag": (_I, [_V, _V, _SZ, _V]),
    "b200_complex_to_mag_squared": (_I, [_V, _V, _SZ, _V]),
    "b200_fir_create": (_I, [C.POINTER(_FirParams), C.POINTER(_V)]),
    "b200_fir_destroy": (_I, [_V]),
    "b200_fir_run": (_I, [_V, _V, _V, _I64, _PI64, _PI64, _V]),
    "b200_fir_run_segment": (_I, [_V, _V, _V, _V, _I64, _PI64, _V]),
    "b200_fir_reset": (_I, [_V, _V]),
    "b200_fir_set_history": (_I, [_V, _V, _V]),
    "b200_fir_get_history": (_I, [_V, _V, _V]),
    "b200_fir_algorithm": (_I, [_V]),
    "b200_fir_geometry": (_I, [_V, C.POINTER(_I), C.POINTER(_I)]),
    "b200_resampler_create": (_I, [C.POINTER(_ResamplerParams), C.POINTER(_V)]),
    "b200_resampler_destroy": (_I, [_V]),
    "b200_resampler_run": (_I, [_V, _V, _V, _I64, _PI64, _PI64, _V]),
    "b200_resampler_run_segment": (_I, [_V, _V, _V, _V, _I64, _PI64, _V]),
    "b200_resampler_reset": (_I, [_V, _V]),
    "b200_resampler_geometry": (_I, [_V, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "b200_fft_create": (_I, [C.POINTER(_FftParams), C.POINTER(_V)]),
    "b200_fft_destroy": (_I, [_V]),
    "b200_fft_run": (_I, [_V, _V, _V, _I64, _V]),
    "b200_fft_geometry": (_I, [_V, C.POINTER(_I), C.POINTER(_I)]),
    "b200_pfb_create": (_I, [C.POINTER(_PfbParams), C.POINTER(_V)]),
    "b200_pfb_destroy": (_I, [_V]),
    "b200_pfb_run": (_I, [_V, _V, _V, _I64, _PI64, _PI64, _V]),
    "b200_pfb_run_segment": (_I, [_V, _V, _V, _V, _I64, _PI64, _V]),
    "b200_pfb_reset": (_I, [_V, _V]),
    "b200_pfb_geometry": (_I, [_V, C.POINTER(_I), C.POINTER(_I)]),
    "b200_pfb_set_algorithm": (_I, [_V, C.c_int32]),
    "b200_pfb_get_algorithm": (_I, [_V, C.POINTER(C.c_int32)]),
    "b200_pfb_get_oversample": (_I, [_V, C.POINTER(C.c_int32)]),
    "b200_chain_create": (_I, [C.POINTER(_ChainOp), C.c_int32, C.c_int32, _I64, C.POINTER(_V)]),
    "b200_chain_destroy": (_I, [_V]),
    "b200_chain_run": (_I, [_V, _V, _V, _I64, _PI64, _V]),
    "b200_chain_run_host": (_I, [_V, _V, _V, _I64, _PI64]),
    "b200_chain_out_bytes_bound": (_I64, [_V, _I64]),
}


def lib() -> C.CDLL:
    """Load the C-ABI library.  Raises (loudly) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise B200Error(f"b200dsp error {rc}: {lib().b200_last_error().decode(errors='replace')}")


def launch_count() -> int:
    return int(lib().b200_launch_count())


def measure_fp32_tflops(iters: int = 4096):
    t, ms = C.c_float(), C.c_float()
    _check(lib().b200_measure_fp32_tflops(int(iters), C.byref(t), C.byref(ms)))
    return float(t.value), float(ms.value)


def measure_fp32x2_tflops(iters: int = 4096):
    t, ms = C.c_float(), C.c_float()
    _check(lib().b200_measure_fp32x2_tflops(int(iters), C.byref(t), C.byref(ms)))
    return float(t.value), float(ms.value)


def _torch():
    import torch
    return torch


def _stream(stream=None) -> int:
    if stream is not None:
        return int(stream)
    return int(_torch().cuda.current_stream().cuda_stream)


def _need_cuda(x):
    if not x.is_cuda:
        raise B200Error("newsched_b200 operates on CUDA tensors only (no CPU fallback)")
    if not x.is_contiguous():
        raise B200Error("tensor must be contiguous")


def _need_out(out, like, numel, dtype=None, what="out"):
    """A caller-supplied output (or halo) goes straight to the kernels as a raw pointer: refuse anything
    that is not a contiguous CUDA tensor of the right dtype / device / size."""
    if not out.is_cuda or out.device != like.device:
        raise B200Error(f"{what} must be a CUDA tensor on {like.device}")
    if not out.is_contiguous():
        raise B200Error(f"{what} must be contiguous")
    if out.dtype != (dtype if dtype is not None else like.dtype):
        raise B200Error(f"{what} has dtype {out.dtype}, expected {dtype if dtype is not None else like.dtype}")
    if out.numel() < numel:
        raise B200Error(f"{what} has {out.numel()} items, needs {numel}")


def _halo_ptr(halo, like, numel):
    """halo: None (zeros), a CUDA tensor, or a raw device pointer (int) -- e.g. a peer-mapped address."""
    if halo is None:
        return None
    if isinstance(halo, int):
        return halo
    _need_out(halo, like, numel, what="halo")
    return halo.data_ptr()


def ipc_export(t) -> bytes:
    """Handle (88 bytes) for the memory of CUDA tensor `t`, importable by another process on the same node."""
    _need_cuda(t)
    h = IpcHandle()
    _check(lib().b200_ipc_export(t.data_ptr(), C.byref(h)))
    return bytes(h)


def ipc_import(raw: bytes) -> int:
    """Maps an exported allocation into this process; returns the device pointer (an int) that aliases the
    exporter's tensor.  Kernels of this GPU read it over NVLink."""
    h = IpcHandle.from_buffer_copy(raw)
    p = C.c_void_p()
    _check(lib().b200_ipc_import(C.byref(h), C.byref(p)))
    return int(p.value)


def ipc_close(raw: bytes, ptr: int) -> None:
    h = IpcHandle.from_buffer_copy(raw)
    _check(lib().b200_ipc_close(C.byref(h), C.c_void_p(ptr)))


def _floats(a):
    import numpy as np
    arr = np.ascontiguousarray(a, dtype=np.float32)
    return arr, arr.ctypes.data_as(C.POINTER(C.c_float))


# --------------------------------------------------------------------- stateless stream blocks
def copy(x, out=None, stream=None):
    """gr::blocks::copy::work (copy.hpp:33-44): bit-exact copy of a CUDA tensor."""
    torch = _torch()
    _need_cuda(x)
    if out is None:
        out = torch.empty_like(x)
    _check(lib().b200_copy(out.data_ptr(), x.data_ptr(), x.numel() * x.element_size(), _stream(stream)))
    return out


def multiply_const(x, k, out=None, stream=None):
    """gr::blocks::multiply_const<T>::work (multiply_const.cpp:19-81); dtype picks ff/cc/ss/ii."""
    torch = _torch()
    _need_cuda(x)
    if out is None:
        out = torch.empty_like(x)
    L, s, n = lib(), _stream(stream), x.numel()
    if x.dtype == torch.float32:
        _check(L.b200_multiply_const_ff(out.data_ptr(), x.data_ptr(), float(k), n, s))
    elif x.dtype == torch.complex64:
        k = complex(k)
        _check(L.b200_multiply_const_cc(out.data_ptr(), x.data_ptr(), k.real, k.imag, n, s))
    elif x.dtype == torch.int16:
        _check(L.b200_multiply_const_ss(out.data_ptr(), x.data_ptr(), int(k), n, s))
    elif x.dtype == torch.int32:
        _check(L.b200_multiply_const_ii(out.data_ptr(), x.data_ptr(), int(k), n, s))
    else:
        raise B200Error(f"multiply_const: unsupported dtype {x.dtype}")
    return out


def _binary(name, a, b, out, stream):
    torch = _torch()
    _need_cuda(a)
    _need_cuda(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        raise B200Error("two-input blocks need equal dtypes and shapes")
    if a.dtype not in (torch.float32, torch.complex64):
        raise B200Error(f"{name}: unsupported dtype {a.dtype}")
    if out is None:
        out = torch.empty_like(a)
    fn = getattr(lib(), f"b200_{name}_{'cc' if a.dtype == torch.complex64 else 'ff'}")
    _check(fn(out.data_ptr(), a.data_ptr(), b.data_ptr(), a.numel(), _stream(stream)))
    return out


def multiply(a, b, out=None, stream=None):
    """Two-input multiply block (float32 or complex64), out = a * b."""
    return _binary("multiply", a, b, out, stream)


def add(a, b, out=None, stream=None):
    """Two-input add block (float32 or complex64), out = a + b."""
    return _binary("add", a, b, out, stream)


def complex_to_mag(x, squared: bool = False, out=None, stream=None):
    torch = _torch()
    _need_cuda(x)
    if x.dtype != torch.complex64:
        raise B200Error("complex_to_mag needs complex64")
    if out is None:
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    fn = lib().b200_complex_to_mag_squared if squared else lib().b200_complex_to_mag
    _check(fn(out.data_ptr(), x.data_ptr(), x.numel(), _stream(stream)))
    return out


# ----------------------------------------------------------------------------- stateful blocks
class FirFilter:
    """fir_filter_ccf / fir_filter_fff, decimating, streaming (history kept on the device)."""

    def __init__(self, taps, decimation: int = 1, is_complex: bool = True, multiply_const=None,
                 algorithm: int = 0):
        arr, ptr = _floats(taps)
        k = complex(multiply_const) if multiply_const is not None else 1 + 0j
        p = _FirParams(ptr, arr.size, int(decimation), int(bool(is_complex)),
                       int(multiply_const is not None), k.real, k.imag, int(algorithm))
        h = C.c_void_p()
        _check(lib().b200_fir_create(C.byref(p), C.byref(h)))
        self._h = h
        self.n_taps, self.decimation, self.is_complex = arr.size, int(decimation), bool(is_complex)
        self.device = _torch().cuda.current_device()     # the handle's buffers live on the device current at create

    @property
    def handle(self):
        return self._h

    @property
    def algorithm(self) -> int:
        return int(lib().b200_fir_algorithm(self._h))

    def _dtype(self):
        torch = _torch()
        return torch.complex64 if self.is_complex else torch.float32

    def work(self, x, out=None, stream=None):
        """One work() call: returns (y, n_consumed).  y has floor(len(x)/D) items."""
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == self._dtype()
        n_out = x.numel() // self.decimation
        if out is None:
            out = torch.empty(n_out, dtype=x.dtype, device=x.device)
        else:
            _need_out(out, x, n_out)
        nc, npd = C.c_int64(), C.c_int64()
        _check(lib().b200_fir_run(self._h, x.data_ptr(), out.data_ptr(), x.numel(), C.byref(nc),
                                  C.byref(npd), _stream(stream)))
        return out[: npd.value], nc.value

    def work_segment(self, x, halo=None, out=None, stream=None):
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == self._dtype()
        n_out = x.numel() // self.decimation
        if out is None:
            out = torch.empty(n_out, dtype=x.dtype, device=x.device)
        else:
            _need_out(out, x, n_out)
        npd = C.c_int64()
        _check(lib().b200_fir_run_segment(self._h, _halo_ptr(halo, x, self.n_taps - 1),
                                          x.data_ptr(), out.data_ptr(), x.numel(), C.byref(npd),
                                          _stream(stream)))
        return out[: npd.value]

    def reset(self, stream=None):
        _check(lib().b200_fir_reset(self._h, _stream(stream)))

    def set_history(self, hist, stream=None):
        assert hist.numel() == self.n_taps - 1
        _check(lib().b200_fir_set_history(self._h, hist.data_ptr(), _stream(stream)))

    def get_history(self, stream=None):
        torch = _torch()
        out = torch.empty(max(self.n_taps - 1, 0), dtype=self._dtype(), device=torch.device("cuda", self.device))
        if self.n_taps > 1:
            _check(lib().b200_fir_get_history(self._h, out.data_ptr(), _stream(stream)))
        return out

    def __del__(self):
        try:
            if self._h:
                lib().b200_fir_destroy(self._h)
                self._h = None
        except Exception:
            pass


class FFT:
    """fft_vcc: N-point complex FFT per item, optional window/shift, fused |.| epilogue and
    fused upstream multiply_const."""

    def __init__(self, n: int, forward: bool = True, window=None, shift: bool = False,
                 output: int = OUT_COMPLEX, pre_multiply_const=None):
        wptr = None
        if window is not None:
            warr, wptr = _floats(window)
            assert warr.size == n
        k = complex(pre_multiply_const) if pre_multiply_const is not None else 1 + 0j
        p = _FftParams(int(n), int(bool(forward)), wptr, int(bool(shift)), int(output),
                       int(pre_multiply_const is not None), k.real, k.imag)
        h = C.c_void_p()
        _check(lib().b200_fft_create(C.byref(p), C.byref(h)))
        self._h = h
        self.n, self.output = int(n), int(output)

    @property
    def handle(self):
        return self._h

    def work(self, x, out=None, stream=None):
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == torch.complex64
        n_vec = x.numel() // self.n
        if out is None:
            dt = torch.complex64 if self.output == OUT_COMPLEX else torch.float32
            out = torch.empty(n_vec * self.n, dtype=dt, device=x.device)
        else:
            _need_out(out, x, n_vec * self.n, torch.complex64 if self.output == OUT_COMPLEX else torch.float32)
        _check(lib().b200_fft_run(self._h, x.data_ptr(), out.data_ptr(), n_vec, _stream(stream)))
        return out

    def __del__(self):
        try:
            if self._h:
                lib().b200_fft_destroy(self._h)
                self._h = None
        except Exception:
            pass


class RationalResampler:
    """rational_resampler_ccf / _fff (interpolation L, decimation D; D = 1 is interp_fir_filter):
    y[m] = sum_k h[k] xu[m*D - k] with xu the L-fold zero-stuffed input.  Streaming: each work()
    consumes whole groups of D items and produces L per group; history lives on the device."""

    def __init__(self, taps, interpolation: int = 1, decimation: int = 1, is_complex: bool = True):
        arr, ptr = _floats(taps)
        p = _ResamplerParams(ptr, arr.size, int(interpolation), int(decimation), int(bool(is_complex)))
        h = C.c_void_p()
        _check(lib().b200_resampler_create(C.byref(p), C.byref(h)))
        self._h = h
        self.n_taps, self.interpolation, self.decimation = arr.size, int(interpolation), int(decimation)
        self.is_complex = bool(is_complex)

    @property
    def handle(self):
        return self._h

    def _n_out(self, n_in):
        return (n_in // self.decimation) * self.interpolation

    def work(self, x, out=None, stream=None):
        """One work() call: returns (y, n_consumed)."""
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == (torch.complex64 if self.is_complex else torch.float32)
        if out is None:
            out = torch.empty(self._n_out(x.numel()), dtype=x.dtype, device=x.device)
        else:
            _need_out(out, x, self._n_out(x.numel()))
        nc, npd = C.c_int64(), C.c_int64()
        _check(lib().b200_resampler_run(self._h, x.data_ptr(), out.data_ptr(), x.numel(), C.byref(nc),
                                        C.byref(npd), _stream(stream)))
        return out[: npd.value], nc.value

    def work_segment(self, x, halo=None, out=None, stream=None):
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == (torch.complex64 if self.is_complex else torch.float32)
        if out is None:
            out = torch.empty(self._n_out(x.numel()), dtype=x.dtype, device=x.device)
        else:
            _need_out(out, x, self._n_out(x.numel()))
        npd = C.c_int64()
        _check(lib().b200_resampler_run_segment(self._h,
                                                _halo_ptr(halo, x, -(-self.n_taps // self.interpolation) - 1),
                                                x.data_ptr(), out.data_ptr(), x.numel(), C.byref(npd),
                                                _stream(stream)))
        return out[: npd.value]

    def reset(self, stream=None):
        _check(lib().b200_resampler_reset(self._h, _stream(stream)))

    def __del__(self):
        try:
            if self._h:
                lib().b200_resampler_destroy(self._h)
                self._h = None
        except Exception:
            pass


class PfbChannelizer:
    """M-channel polyphase analysis bank, one output frame per hop = M / oversample input items;
    work() returns [n_t, channels]."""

    def __init__(self, taps, n_channels: int, channel_begin: int = 0, channel_count: int = 0,
                 algorithm: int = 0, oversample: int = 1):
        """algorithm: 0 auto, 1 SIMT DFT, 2 DFT across branches as a tensor-core GEMM (64 channels only).
        oversample: 1 critically sampled, 2 or 4 (M = 16 .. 256; see b200_pfb_params in include/b200dsp.h)."""
        arr, ptr = _floats(taps)
        assert arr.size % n_channels == 0
        p = _PfbParams(ptr, int(n_channels), arr.size // n_channels, int(channel_begin), int(channel_count),
                       int(oversample))
        h = C.c_void_p()
        _check(lib().b200_pfb_create(C.byref(p), C.byref(h)))
        self._h = h
        if algorithm:
            try:
                _check(lib().b200_pfb_set_algorithm(self._h, int(algorithm)))
            except Exception:
                lib().b200_pfb_destroy(self._h)
                self._h = None
                raise
        self.m = int(n_channels)
        self.p = arr.size // n_channels
        self.channels = int(channel_count) if channel_count else self.m - int(channel_begin)
        self.oversample = self._get_oversample()
        self.hop = self.m // self.oversample

    @property
    def handle(self):
        return self._h

    @property
    def algorithm(self) -> int:
        a = C.c_int32()
        _check(lib().b200_pfb_get_algorithm(self._h, C.byref(a)))
        return a.value

    def _get_oversample(self) -> int:
        v = C.c_int32()
        _check(lib().b200_pfb_get_oversample(self._h, C.byref(v)))
        return v.value

    def work(self, x, out=None, stream=None):
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == torch.complex64
        n_t = x.numel() // self.hop
        if out is None:
            out = torch.empty((n_t, self.channels), dtype=torch.complex64, device=x.device)
        else:
            _need_out(out, x, n_t * self.channels)
        nc, nv = C.c_int64(), C.c_int64()
        _check(lib().b200_pfb_run(self._h, x.data_ptr(), out.data_ptr(), x.numel(), C.byref(nc),
                                  C.byref(nv), _stream(stream)))
        return out[: nv.value], nc.value

    def work_segment(self, x, halo=None, out=None, stream=None):
        torch = _torch()
        _need_cuda(x)
        assert x.dtype == torch.complex64
        n_t = x.numel() // self.hop
        if out is None:
            out = torch.empty((n_t, self.channels), dtype=torch.complex64, device=x.device)
        else:
            _need_out(out, x, n_t * self.channels)
        nv = C.c_int64()
        _check(lib().b200_pfb_run_segment(self._h, _halo_ptr(halo, x, self.p * self.m - self.hop),
                                          x.data_ptr(), out.data_ptr(), x.numel(), C.byref(nv),
                                          _stream(stream)))
        return out[: nv.value]

    def reset(self, stream=None):
        _check(lib().b200_pfb_reset(self._h, _stream(stream)))

    def __del__(self):
        try:
            if self._h:
                lib().b200_pfb_destroy(self._h)
                self._h = None
        except Exception:
            pass


class Chain:
    """Ordered list of ops run back to back on device buffers.

    ops: list of ("copy",) | ("multiply_const_cc", k) | ("multiply_const_ff", k) |
         ("complex_to_mag",) | FirFilter | FFT | PfbChannelizer
    """

    def __init__(self, ops, in_item_bytes: int = 8, chunk_items: int = 1 << 24):
        arr = (_ChainOp * len(ops))()
        self._keep = list(ops)
        for i, op in enumerate(ops):
            if isinstance(op, FirFilter):
                arr[i] = _ChainOp(OP_FIR, op.handle, 0.0, 0.0)
            elif isinstance(op, FFT):
                arr[i] = _ChainOp(OP_FFT, op.handle, 0.0, 0.0)
            elif isinstance(op, PfbChannelizer):
                arr[i] = _ChainOp(OP_PFB, op.handle, 0.0, 0.0)
            elif op[0] == "copy":
                arr[i] = _ChainOp(OP_COPY, None, 0.0, 0.0)
            elif op[0] == "multiply_const_cc":
                k = complex(op[1])
                arr[i] = _ChainOp(OP_MULTIPLY_CONST_CC, None, k.real, k.imag)
            elif op[0] == "multiply_const_ff":
                arr[i] = _ChainOp(OP_MULTIPLY_CONST_FF, None, float(op[1]), 0.0)
            elif op[0] == "complex_to_mag":
                arr[i] = _ChainOp(OP_COMPLEX_TO_MAG, None, 0.0, 0.0)
            else:
                raise B200Error(f"unknown chain op {op!r}")
        h = C.c_void_p()
        _check(lib().b200_chain_create(arr, len(ops), int(in_item_bytes), int(chunk_items), C.byref(h)))
        self._h = h
        self.in_item_bytes = int(in_item_bytes)

    def out_bytes(self, n_in_items: int) -> int:
        return int(lib().b200_chain_out_bytes_bound(self._h, int(n_in_items)))

    def run(self, x, out, stream=None) -> int:
        """Device-resident pass; `out` is a uint8/any CUDA tensor big enough.  Returns bytes written."""
        _need_cuda(x)
        _need_cuda(out)
        n_items = x.numel() * x.element_size() // self.in_item_bytes
        if out.device != x.device or out.numel() * out.element_size() < self.out_bytes(n_items):
            raise B200Error(f"Chain.run: out must be on {x.device} with >= {self.out_bytes(n_items)} bytes")
        nb = C.c_int64()
        _check(lib().b200_chain_run(self._h, x.data_ptr(), out.data_ptr(), n_items, C.byref(nb),
                                    _stream(stream)))
        return nb.value

    def run_host(self, x_host, out_host) -> int:
        """Host-resident pass (pinned CPU tensors): H2D, compute and D2H overlapped.  Blocking."""
        if x_host.is_cuda or out_host.is_cuda:
            raise B200Error("run_host takes host (pinned) tensors")
        n_items = x_host.numel() * x_host.element_size() // self.in_item_bytes
        if not (x_host.is_contiguous() and out_host.is_contiguous()) or \
                out_host.numel() * out_host.element_size() < self.out_bytes(n_items):
            raise B200Error(f"Chain.run_host: contiguous host tensors, out >= {self.out_bytes(n_items)} bytes")
        nb = C.c_int64()
        _check(lib().b200_chain_run_host(self._h, x_host.data_ptr(), out_host.data_ptr(), n_items,
                                         C.byref(nb)))
        return nb.value

    def __del__(self):
        try:
            if self._h:
                lib().b200_chain_destroy(self._h)
                self._h = None
        except Exception:
            pass


class DeviceRing:
    """Doubly mapped device ring (CUDA VMM): base[i] aliases base[i + size]."""

    def __init__(self, min_bytes: int):
        h = C.c_void_p()
        _check(lib().b200_ring_create(int(min_bytes), C.byref(h)))
        self._h = h
        self.base = int(lib().b200_ring_base(h))
        self.size = int(lib().b200_ring_size(h))

    def __del__(self):
        try:
            if self._h:
                lib().b200_ring_destroy(self._h)
                self._h = None
        except Exception:
            pass
