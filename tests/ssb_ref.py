"""Single-sideband output (``-m usb`` / ``-m lsb``): its oracle (TEST INFRASTRUCTURE).

Per row, on the decimator output ``y`` that ``re`` / ``im`` / ``iq`` read: the prototype
``h = ellip(3, 1, 30, B/2)`` at ``fs_d = fs // q`` (B = omegaOut), ``Omega = +-pi B / fs_d`` and
``s[k] = Re(e^{j Omega k} sosfilt(h, y e^{-j Omega k})[k])`` from a zero state: per chunk in the
default mode, once over the whole stream in seamless mode.
"""
import numpy as np
from scipy import signal

from oracle import oracle as orc


def ssb_sos(fs: int, q: int, B: int) -> np.ndarray:
    """The prototype low-pass, the fm/am output filter's design call at half the width."""
    return signal.ellip(3, 1, 30, B / 2, btype='lowpass', output='sos', fs=fs // q)


def ssb_omega(demod: str, B: int, fs_d: int) -> float:
    om = np.pi * B / fs_d
    return om if demod == 'usb' else -om


def ssb(y: np.ndarray, sos: np.ndarray, omega: float) -> np.ndarray:
    """Re(e^{j omega k} sosfilt(sos, y e^{-j omega k})) along the last axis, k from 0."""
    y = np.asarray(y, dtype=np.complex128)
    rot = np.exp(1j * omega * np.arange(y.shape[-1]))
    return np.real(rot * signal.sosfilt(sos, y * np.conj(rot), axis=-1))


def _params(kw: dict):
    return ssb_sos(kw['fs'], kw['dec'], kw['omega_out']), ssb_omega(kw['demod'], kw['omega_out'], kw['fs'] // kw['dec'])


def ssb_oracle(kw: dict, stream: bytes) -> np.ndarray:
    """Chunk-local usb / lsb output of a byte stream, (R, C*M): every chunk from a zero state."""
    sos, om = _params(kw)
    ch = orc.Chain(**{**kw, 'demod': 're'})
    st = np.frombuffer(stream, dtype=np.uint8)
    zs = [ch.ingest(st[o:o + ch.chunk_bytes]).copy() for o in range(0, st.size, ch.chunk_bytes)]
    if not zs:
        return np.empty((ch.R, 0), dtype=np.float64)
    y = ch.decimated(np.stack(zs))                       # (C, R, M)
    s = ssb(y, sos, om)
    return np.ascontiguousarray(s.transpose(1, 0, 2)).reshape(ch.R, -1)


def seamless_ssb_oracle(kw: dict, stream: bytes) -> tuple[np.ndarray, complex]:
    """Seamless usb / lsb output (R, C*M) of a whole-chunk stream (one filter over the stream), and
    the final IQ offset."""
    from seamless_ref import seamless_decimated
    sos, om = _params(kw)
    y, off = seamless_decimated({**kw, 'demod': 're'}, stream)
    return ssb(y, sos, om), off
