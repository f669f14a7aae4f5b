"""Module-level operators of the reference's ``src/dsp/demodulation.py`` (:25-79), same names and
calling convention -- the caller owns both arrays, results are written in place, nothing is
returned -- executed by the CUDA library (``sdrb_fm_demod`` .. ``sdrb_shift_freq`` of
include/sdrterm_b200.h).  There is no CPU implementation here."""
from __future__ import annotations

import numpy as np

from .. import _native as nat

__all__ = ['fmDemod', 'amDemod', 'realOutput', 'imagOutput', 'iqOutput', 'ssbDemod', 'usbDemod', 'lsbDemod',
           'shiftFreq']


def _rows(data, out):
    d = np.ascontiguousarray(np.atleast_2d(data), dtype=np.complex128)
    if not isinstance(out, np.ndarray):
        raise TypeError('output must be a numpy array')
    o2 = np.atleast_2d(out)
    if o2.shape != d.shape:
        raise ValueError(f'output shape {o2.shape} does not match input shape {d.shape}')
    return d, o2


def _run(entry: str, data, out, device: int = 0) -> None:
    d, o2 = _rows(data, out)
    res = np.empty(d.shape, dtype=np.float64)
    fn = getattr(nat.lib(), entry)
    nat.check(fn(device, d.ctypes.data, d.shape[0], d.shape[1], res.ctypes.data))
    o2[...] = res


def fmDemod(data, tmp) -> None:
    """``tmp[r] = resample(angle(data[r, 0::2] * conj(data[r, 1::2])), n)`` (demodulation.py:25-38)."""
    _run('sdrb_fm_demod', data, tmp)


def amDemod(data, res) -> None:
    """``res = abs(square(data))`` (demodulation.py:41-48)."""
    _run('sdrb_am_demod', data, res)


def realOutput(data, res) -> None:
    """``res = real(data)`` (demodulation.py:51-58)."""
    _run('sdrb_real_output', data, res)


def imagOutput(data, res) -> None:
    """``res = imag(data)`` (demodulation.py:61-68)."""
    _run('sdrb_imag_output', data, res)


def iqOutput(data, res) -> None:
    """``res[r, 2k] = real(data[r, k])``, ``res[r, 2k+1] = imag(data[r, k])``: the complex rows as
    interleaved doubles, ``res`` shaped (R, 2M).  Not a reference operator (``-m iq``)."""
    d = np.ascontiguousarray(np.atleast_2d(data), dtype=np.complex128)
    if not isinstance(res, np.ndarray):
        raise TypeError('output must be a numpy array')
    o2 = np.atleast_2d(res)
    if o2.shape != (d.shape[0], 2 * d.shape[1]):
        raise ValueError(f'output shape {o2.shape} does not match (R, 2M) = {(d.shape[0], 2 * d.shape[1])}')
    out = np.empty(o2.shape, dtype=np.float64)
    nat.check(nat.lib().sdrb_iq_output(0, d.ctypes.data, d.shape[0], d.shape[1], out.ctypes.data))
    o2[...] = out


def ssbDemod(data, res, sos, omega: float) -> None:
    """Single-sideband demodulation, ``res`` shaped like ``data``: per row, from a zero filter state,
    ``res[k] = real(exp(1j*omega*k) * sosfilt(sos, data * exp(-1j*omega*k))[k])`` -- the prototype
    low-pass ``sos`` (1..4 sections) moved to a complex band-pass around ``omega`` (rad/sample,
    0 < |omega| < pi/2; > 0 keeps the upper sideband, < 0 the lower).  Not a reference operator
    (``-m usb`` / ``-m lsb``)."""
    d, o2 = _rows(data, res)
    s = np.ascontiguousarray(sos, dtype=np.float64).reshape(-1, 6)
    out = np.empty(d.shape, dtype=np.float64)
    nat.check(nat.lib().sdrb_ssb_demod(0, d.ctypes.data, d.shape[0], d.shape[1], s.ctypes.data, s.shape[0],
                                       float(omega), out.ctypes.data))
    o2[...] = out


def usbDemod(data, res, sos, omega: float) -> None:
    """``ssbDemod`` for the upper sideband (``omega > 0``): the operator ``-m usb`` selects."""
    if not omega > 0:
        raise ValueError('the upper sideband needs omega > 0')
    ssbDemod(data, res, sos, omega)


def lsbDemod(data, res, sos, omega: float) -> None:
    """``ssbDemod`` for the lower sideband (``omega < 0``): the operator ``-m lsb`` selects."""
    if not omega < 0:
        raise ValueError('the lower sideband needs omega < 0')
    ssbDemod(data, res, sos, omega)


def shiftFreq(y, shift, res) -> None:
    """``res[m, n] = y[n] * shift[m, n]`` (demodulation.py:71-79)."""
    yv = np.ascontiguousarray(y, dtype=np.complex128).reshape(-1)
    sh = np.ascontiguousarray(np.atleast_2d(shift), dtype=np.complex128)
    if sh.shape[1] != yv.size or np.atleast_2d(res).shape != sh.shape:
        raise ValueError('shiftFreq: shapes (n), (m,n) -> (m,n) expected')
    out = np.empty(sh.shape, dtype=np.complex128)
    nat.check(nat.lib().sdrb_shift_freq(0, yv.ctypes.data, sh.ctypes.data, sh.shape[0], sh.shape[1],
                                        out.ctypes.data))
    np.atleast_2d(res)[...] = out
