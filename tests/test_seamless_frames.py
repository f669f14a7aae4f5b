"""CPU: the seamless frame (plan.seamless_frame_samples) and the frame plans of any decimation."""
import pytest

from sdrterm_b200.plan import CHUNK_BYTES, build_plan, lookahead_chunks, seamless_frame_samples

_ISZ = {'B': 1, 'h': 2, 'f': 4, 'd': 8}


@pytest.mark.parametrize('enc,q,Nf,Mf,tiles', [('B', 50, 64000, 1280, 40), ('h', 25, 32000, 1280, 40),
                                               ('h', 3, 32736, 10912, 341), ('f', 100, 16000, 160, 5),
                                               ('d', 255, 8160, 32, 1)])
def test_frame_table(enc, q, Nf, Mf, tiles):
    N = CHUNK_BYTES // (2 * _ISZ[enc])
    assert seamless_frame_samples(N, q) == Nf
    assert Nf // q == Mf and Mf // 32 == tiles and Nf % (32 * q) == 0


def test_frames_are_chunks_for_powers_of_two():
    for enc, isz in _ISZ.items():
        N = CHUNK_BYTES // (2 * isz)
        for k in range(1, 20):
            q = 1 << k
            if N % (32 * q) == 0:
                assert seamless_frame_samples(N, q) == N


@pytest.mark.parametrize('q', [3, 5, 25, 50, 100, 255])
def test_frame_plan_builds(q):
    N = CHUNK_BYTES // 2
    Nf = seamless_frame_samples(N, q)
    pl = build_plan(2_400_000, 'B', q, [0], correct_iq=True, demod='re', seamless=True, chunk_bytes=2 * Nf)
    assert pl.N == Nf and pl.rem == 0 and pl.cnt_last == 32 and pl.ntiles == Nf // (32 * q)
    assert pl.lookahead == lookahead_chunks(pl.modes.p, pl.modes.rho_p, Nf)
    with pytest.raises(ValueError, match='divide'):
        build_plan(2_400_000, 'B', q, [0], demod='re', seamless=True)


# ------------------------------------------------------------------------------------------------
# The numpy twin of frames and the ragged end (tests/frames_ref.py) against the seamless oracle.
import numpy as np  # noqa: E402

import signals  # noqa: E402
from frames_ref import FrameTwin, ragged_oracle  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from seamless_ref import seamless_oracle  # noqa: E402
from util import rel_err  # noqa: E402


def _kw(enc, q, demod, iq, center, fs):
    return dict(fs=fs, enc=enc, center=center, dec=q, demod=demod, omega_out=5000, correct_iq=iq, vfos=None,
                simo=False, normalize=False, swap=False, big_endian=None)


def _frame_plan(kw):
    ch = orc.Chain(**kw)
    sb = 2 * _ISZ[kw['enc']]
    nf = seamless_frame_samples(CHUNK_BYTES // sb, kw['dec'])
    return build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, correct_iq=kw['correct_iq'], demod=kw['demod'],
                      omega_out=kw['omega_out'], seamless=True, chunk_bytes=nf * sb)


def _twin(pl, body, split):
    tw = FrameTwin(pl)
    sb = pl.chunk_bytes // pl.N
    outs = [tw.stream_samples(body[o:o + split * sb]) for o in range(0, len(body), split * sb)]
    return np.concatenate(outs + [tw.end()], axis=1)


@pytest.mark.parametrize('name,kw,nbytes', [
    # uint8 -d 50 (config 2): two frames, then Lp = 3072 (61 full blocks and 22 samples)
    ('uint8 d50 am iq', _kw('B', 50, 'am', True, -20000, 2_400_000), 2 * CHUNK_BYTES),
    # int16 -d 3: one frame of 32736, then Lp = 32
    ('int16 d3 re', _kw('h', 3, 're', False, 30000, 240_000), CHUNK_BYTES),
    # float64 -d 255: one frame of 8160, then Lp = 32 < q: Mf' = 0, one output from the partial block
    ('float64 d255 im iq', _kw('d', 255, 'im', True, 12000, 2_400_000), CHUNK_BYTES),
    # uint8 -d 50 fm ending 10 samples after a frame: the end window reaches into the frame before
    ('uint8 d50 fm Lp10', _kw('B', 50, 'fm', True, -20000, 2_400_000), 2 * 64010),
])
def test_frame_twin_matches_oracle(name, kw, nbytes):
    pl = _frame_plan(kw)
    body = signals.generic_bytes(kw['enc'], CHUNK_BYTES // (2 * _ISZ[kw['enc']]) * 2, 41, kw['fs'],
                                 kw['center'] or 40_000)[:nbytes]
    ref = seamless_oracle(kw, body)[0] if nbytes % CHUNK_BYTES == 0 else ragged_oracle(kw, body)
    out = _twin(pl, body, 7001)
    err = rel_err(out, ref)
    L = nbytes // (pl.chunk_bytes // pl.N)
    print(f'{name}: N_f={pl.N} L={L} Lp={L % pl.N} outputs={out.shape[1]} err={err:.3e}')
    assert out.shape == ref.shape and out.shape[1] == -(-L // pl.q)
    assert err < 1e-11
    assert rel_err(_twin(pl, body, pl.N + 3), out) < 1e-13


@pytest.mark.parametrize('L', [1, 20, 27])
def test_short_streams_refused(L):
    """At most 27 samples (the decimator's pad): SciPy refuses the stream, and so does the seamless
    end (the twin here, SDRB_ERR_ARG on the handle, tests/test_gpu_seamless_frames.py)."""
    kw = _kw('B', 50, 'am', False, 0, 2_400_000)
    pl = _frame_plan(kw)
    assert pl.edge == 27
    body = signals.generic_bytes('B', 64, 3, kw['fs'], 40_000)[:2 * L]
    z = np.frombuffer(body, dtype=np.uint8).astype(float)
    with pytest.raises(ValueError):
        signal_decimate(z[0::2] + 1j * z[1::2], 50)
    tw = FrameTwin(pl)
    tw.stream_samples(body)
    with pytest.raises(ValueError):
        tw.end()


def signal_decimate(x, q):
    from scipy import signal
    return signal.decimate(x, q)
