"""Complex baseband output (``-m iq``): its oracle (TEST INFRASTRUCTURE).

The iq output of a chunk and row is the decimator output ``y`` of ``oracle.Chain`` (chunk-local
mode) or of ``seamless_ref.seamless_decimated`` (seamless mode) written as interleaved doubles:
``out[r, c*2M + 2k] = Re y[c, r, k]``, ``out[r, c*2M + 2k + 1] = Im y[c, r, k]``.  There is no
output low-pass, exactly as for ``re`` / ``im``.
"""
import numpy as np

from oracle import oracle as orc


def interleave(re: np.ndarray, im: np.ndarray) -> np.ndarray:
    """(R, C*M) real and imaginary rows -> (R, C*2M) with (Re, Im) per output."""
    re = np.asarray(re, dtype=np.float64)
    out = np.empty((re.shape[0], 2 * re.shape[1]), dtype=np.float64)
    out[:, 0::2] = re
    out[:, 1::2] = im
    return out


def _complex_rows(y: np.ndarray) -> np.ndarray:
    """(R, K) complex -> (R, 2K) interleaved doubles."""
    return np.ascontiguousarray(y, dtype=np.complex128).view(np.float64).reshape(y.shape[0], -1)


def iq_oracle(kw: dict, stream: bytes) -> np.ndarray:
    """Chunk-local iq output of a byte stream, (R, C*2M), read chunk by chunk like ``Chain.run``."""
    ch = orc.Chain(**{**kw, 'demod': 're'})
    st = np.frombuffer(stream, dtype=np.uint8)
    zs = [ch.ingest(st[o:o + ch.chunk_bytes]).copy() for o in range(0, st.size, ch.chunk_bytes)]
    if not zs:
        return np.empty((ch.R, 0), dtype=np.float64)
    y = ch.decimated(np.stack(zs))                       # (C, R, M)
    return _complex_rows(np.ascontiguousarray(y.transpose(1, 0, 2)).reshape(ch.R, -1))


def seamless_iq_oracle(kw: dict, stream: bytes) -> tuple[np.ndarray, complex]:
    """Seamless iq output (R, C*2M) of a whole-chunk stream, and the final IQ offset."""
    from seamless_ref import seamless_decimated
    y, off = seamless_decimated(kw, stream)
    return _complex_rows(y), off
