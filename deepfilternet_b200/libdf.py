"""Drop-in for the reference's PyO3 module ``libdf`` (pyDF/src/lib.rs, stubs pyDF/libdf.pyi):
class ``DF`` plus ``erb``, ``erb_inv``, ``erb_norm``, ``unit_norm``, ``unit_norm_init`` -- same
names, argument meaning, return types (numpy arrays) and error behaviour, computed by the CUDA
kernels of libdfb200.so through its C ABI (host-pointer entry points).

Differences kept on purpose (documented in INTEGRATION.md):
  * ``DF.synthesis`` / ``erb_norm`` do not clobber their inputs (the reference mutates them through
    ``unsafe as_array_mut``, pyDF/src/lib.rs:87,262);
  * ``reset=False`` carries the STFT / ISTFT memories across calls and channels exactly like the
    reference's shared ``DFState`` (channel 0 continues the previous call, channel c continues c - 1);
  * STFT geometries: 960 / 480 (every shipped model) runs specialised kernels; any other even
    fft_size with 32 <= fft_size <= 4096 and no prime factor above 7 in fft_size / 2 (320, 384,
    512, 640, 882, 1024, 1920, 4096, ...) runs the runtime mixed-radix kernels, for every
    hop_size <= fft_size / 2.  Other sizes raise ``DfbError`` (DFB_ERR_UNSUPPORTED).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from ._lib import DfbError, check

_DEVICE = 0


def set_device(device: int) -> None:
    """CUDA ordinal used by the module-level functions and new ``DF`` objects."""
    global _DEVICE
    _DEVICE = int(device)


def _ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def _require(a: np.ndarray):
    if a.size == 0 or not a.flags["C_CONTIGUOUS"]:
        # pyDF/src/lib.rs:59-64
        raise RuntimeError("[df] Input array empty or not contiguous.")


def _wrap(rc: int):
    try:
        check(rc)
    except DfbError as e:
        if e.code == _lib.DFB_ERR_INVALID:
            raise RuntimeError(f"DF shape error: {e}") from None
        raise


class DF:
    """pyDF ``DF`` (pyDF/src/lib.rs:14-136)."""

    def __init__(self, sr: int, fft_size: int, hop_size: int, nb_bands: Optional[int] = 32,
                 min_nb_erb_freqs: Optional[int] = 1, device: Optional[int] = None):
        nb_bands = 32 if nb_bands is None else int(nb_bands)
        min_nb_erb_freqs = 1 if min_nb_erb_freqs is None else int(min_nb_erb_freqs)
        self._device = _DEVICE if device is None else int(device)
        self._sr, self._fft, self._hop, self._nb = int(sr), int(fft_size), int(hop_size), nb_bands
        self._min_nb = min_nb_erb_freqs
        if self._hop * 2 > self._fft:
            # the reference panics (PanicException) at libDF/src/lib.rs:111
            raise RuntimeError("assertion failed: hop_size * 2 <= fft_size")
        h = C.c_void_p()
        check(_lib.lib().dfb_state_create(C.byref(h), self._device, self._sr, self._fft, self._hop,
                                          nb_bands, min_nb_erb_freqs))
        self._h = h

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                _lib.lib().dfb_state_free(h)
            except Exception:
                pass
            self._h = None

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    @property
    def device(self) -> int:
        return self._device

    def analysis(self, input: np.ndarray, reset: Optional[bool] = True) -> np.ndarray:
        """f32[C,T] -> c64[C, T // hop, fft // 2 + 1]  (pyDF/src/lib.rs:41-72)"""
        x = np.asarray(input)
        if x.dtype != np.float32 or x.ndim != 2:
            raise TypeError("argument 'input': expected a 2-D float32 numpy array")
        _require(x)
        c, t = x.shape
        out = np.empty((c, t // self._hop, self._fft // 2 + 1), dtype=np.complex64)
        if out.size:
            check(_lib.lib().dfb_analysis_host_ex(self._h, _ptr(x), c, t, 1 if (reset is None or reset) else 0, _ptr(out)))
        return out

    def synthesis(self, input: np.ndarray, reset: Optional[bool] = True) -> np.ndarray:
        """c64[C,T',F] -> f32[C, T' * hop]  (pyDF/src/lib.rs:74-107)"""
        x = np.asarray(input)
        if x.dtype != np.complex64 or x.ndim != 3:
            raise TypeError("argument 'input': expected a 3-D complex64 numpy array")
        _require(x)
        c, tf, f = x.shape
        if f != self._fft // 2 + 1:
            raise RuntimeError(f"DF shape error: expected {self._fft // 2 + 1} frequency bins, got {f}")
        out = np.empty((c, tf * self._hop), dtype=np.float32)
        check(_lib.lib().dfb_synthesis_host_ex(self._h, _ptr(x), c, tf, 1 if (reset is None or reset) else 0, _ptr(out)))
        return out

    def erb_widths(self) -> np.ndarray:
        out = np.zeros(self._nb, dtype=np.int64)
        check(_lib.lib().dfb_state_erb_widths(self._h, out.ctypes.data_as(C.POINTER(C.c_int64))))
        return out.astype(np.uint64)

    def fft_window(self) -> np.ndarray:
        out = np.zeros(self._fft, dtype=np.float32)
        check(_lib.lib().dfb_state_fft_window(self._h, out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def sr(self) -> int:
        return self._sr

    def fft_size(self) -> int:
        return self._fft

    def hop_size(self) -> int:
        return self._hop

    def nb_erb(self) -> int:
        return self._nb

    def reset(self) -> None:
        check(_lib.lib().dfb_state_reset(self._h))


def _widths(erb_fb) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(erb_fb).astype(np.int64))


def _lead_dims(x: np.ndarray, what: str):
    if x.ndim not in (2, 3, 4):
        # pyDF/src/lib.rs:162-166, 220-224
        raise ValueError(f"Dimension not supported for {what}: {x.ndim}")


def erb(input: np.ndarray, erb_fb: np.ndarray, db: Optional[bool] = True) -> np.ndarray:
    """c64[..., F] -> f32[..., E]  (pyDF/src/lib.rs:142-192)"""
    x = np.ascontiguousarray(input, dtype=np.complex64)
    _lead_dims(x, "erb")
    _require(x)
    fb = _widths(erb_fb)
    f = x.shape[-1]
    out = np.empty(x.shape[:-1] + (len(fb),), dtype=np.float32)
    _wrap(_lib.lib().dfb_erb_host(_DEVICE, _ptr(x), x.size // f, f, fb.ctypes.data_as(C.POINTER(C.c_int64)),
                                  len(fb), 1 if (db is None or db) else 0, _ptr(out)))
    return out


def erb_inv(input: np.ndarray, erb_fb: np.ndarray) -> np.ndarray:
    """f32[..., E] -> f32[..., sum(erb_fb)]  (pyDF/src/lib.rs:194-250)"""
    x = np.ascontiguousarray(input, dtype=np.float32)
    fb = _widths(erb_fb)
    if x.shape[-1] != len(fb):
        raise ValueError(f"Number of erb bands do not match with input: {x.shape[-1]}, {len(fb)}")
    _lead_dims(x, "erb")
    _require(x)
    out = np.empty(x.shape[:-1] + (int(fb.sum()),), dtype=np.float32)
    _wrap(_lib.lib().dfb_erb_inv_host(_DEVICE, _ptr(x), x.size // len(fb),
                                      fb.ctypes.data_as(C.POINTER(C.c_int64)), len(fb), _ptr(out)))
    return out


def erb_norm(erb: np.ndarray, alpha: float, state: Optional[np.ndarray] = None) -> np.ndarray:
    """f32[C,T,E] -> f32[C,T,E]  (pyDF/src/lib.rs:252-274)"""
    x = np.ascontiguousarray(erb, dtype=np.float32)
    if x.ndim != 3:
        raise TypeError("argument 'erb': expected a 3-D float32 numpy array")
    _require(x)
    st = None
    if state is not None:
        st = np.ascontiguousarray(state, dtype=np.float32)
        if st.shape != (x.shape[0], x.shape[2]):
            raise RuntimeError(f"DF shape error: state shape {st.shape} != {(x.shape[0], x.shape[2])}")
    out = np.empty_like(x)
    _wrap(_lib.lib().dfb_erb_norm_host(_DEVICE, _ptr(x), x.shape[0], x.shape[1], x.shape[2], float(alpha),
                                       _ptr(st) if st is not None else None, _ptr(out)))
    return out


def unit_norm(spec: np.ndarray, alpha: float, state: Optional[np.ndarray] = None) -> np.ndarray:
    """c64[C,T,F] -> c64[C,T,F]  (pyDF/src/lib.rs:276-298)"""
    x = np.ascontiguousarray(spec, dtype=np.complex64)
    if x.ndim != 3:
        raise TypeError("argument 'spec': expected a 3-D complex64 numpy array")
    _require(x)
    st = None
    if state is not None:
        st = np.ascontiguousarray(state, dtype=np.float32)
        if st.shape != (x.shape[0], x.shape[2]):
            raise RuntimeError(f"DF shape error: state shape {st.shape} != {(x.shape[0], x.shape[2])}")
    out = np.empty_like(x)
    _wrap(_lib.lib().dfb_unit_norm_host(_DEVICE, _ptr(x), x.shape[0], x.shape[1], x.shape[2], float(alpha),
                                        _ptr(st) if st is not None else None, _ptr(out)))
    return out


def unit_norm_init(num_freq_bins: int) -> np.ndarray:
    """-> f32[1, n] = linspace(0.001, 0.0001, n)  (pyDF/src/lib.rs:300-307)"""
    out = np.empty((1, int(num_freq_bins)), dtype=np.float32)
    check(_lib.lib().dfb_unit_norm_init(int(num_freq_bins), _ptr(out)))
    return out
