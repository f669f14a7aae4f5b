"""CPU: the seamless streaming mode without a device -- the seamless oracle pinned against the
chunk-local oracle, the numpy twin of the seamless finish stage (tests/seamless_ref.py) against the
oracle, the lookahead D and the plan's refusals."""
import numpy as np
import pytest
from scipy import signal

import seamless_ref as S
import signals
from oracle import oracle as orc
from sdrterm_b200.plan import build_plan, filter_modes, lookahead_bound, lookahead_chunks, LOOKAHEAD_TOL
from util import rel_err

_ISZ = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'f': 4, 'd': 8}


def _kw(enc, q, demod, iq, center, fs=1_024_000, simo=False, vfos=None, swap=False, omega=5000):
    return dict(fs=fs, enc=enc, center=center, dec=q, demod=demod, omega_out=omega, correct_iq=iq, vfos=vfos,
                simo=simo, normalize=False, swap=swap, big_endian=None)


def _plan(kw):
    ch = orc.Chain(**kw)
    return build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, simo=kw['simo'], swap=orc.needs_swap(ch.dt),
                      correct_iq=kw['correct_iq'], normalize=kw['normalize'], demod=kw['demod'],
                      omega_out=kw['omega_out'], seamless=True)


def _body(kw, nch, seed):
    n = nch * 131072 // (2 * _ISZ[kw['enc']])
    if kw['simo']:
        return signals.c3_bytes(n, seed=3)[0]
    return signals.generic_bytes(kw['enc'], n, seed, kw['fs'], kw['center'] or 40_000, big_endian=kw['swap'])


@pytest.mark.parametrize('demod', ['am', 're', 'im'])
def test_one_chunk_oracle_equals_chunk_local_oracle(demod):
    """On a one-chunk stream the two contracts differ only by the NCO phase: exact integer phase
    here, the reference's rounded phase increment there (at most ~N ulps of phase)."""
    kw = _kw('h', 64, demod, True, 15000)
    body = _body(kw, 1, 1)
    ref, _ = S.seamless_oracle(kw, body)
    loc = orc.Chain(**kw).run(body)
    err = rel_err(ref, loc)
    print(f'{demod}: seamless vs chunk-local oracle on one chunk {err:.2e}')
    assert err < 1e-11


def test_discriminator_even_samples_are_the_reference_pair_phases():
    kw = _kw('h', 64, 'fm', True, 15000)
    body = _body(kw, 1, 2)
    y, _ = S.seamless_decimated(kw, body)
    ch = orc.Chain(**kw)
    yl = ch.decimated(ch.ingest(np.frombuffer(body, dtype=np.uint8)).copy()[None])[0]
    d = S.discriminator(y)
    pairs = np.angle(yl[:, 0::2] * np.conj(yl[:, 1::2]))
    assert np.max(np.abs(d[:, 0::2] - pairs)) / np.max(np.abs(pairs)) < 1e-11


def test_seamless_oracle_is_scipy_on_the_whole_stream():
    kw = _kw('B', 8, 'am', False, -20000, fs=2_400_000)
    body = _body(kw, 2, 3)
    ref, _ = S.seamless_oracle(kw, body)
    z = orc.decode(np.frombuffer(body, dtype=np.uint8), orc.sample_dtype('B'))
    u = z * np.exp(-2j * np.pi * (((-20000 * np.arange(z.size)) % 2_400_000) / 2_400_000))
    y = signal.decimate(u, 8)
    sos = orc.output_filter_sos(2_400_000 // 8, 5000)
    assert rel_err(ref, signal.sosfilt(sos, np.abs(y * y))[None]) < 1e-13


TWIN = [
    ('int16 d64 fm iq', _kw('h', 64, 'fm', True, 15000), 4, (1, 2)),
    ('int16 d64 am centre0', _kw('h', 64, 'am', False, 0), 3, (2, 1)),
    ('int16 d64 re iq', _kw('h', 64, 're', True, 15000), 3, (3,)),
    ('int16 d64 im', _kw('h', 64, 'im', False, -9000), 3, (1,)),
    ('uint8 d8 am iq', _kw('B', 8, 'am', True, -20000, fs=2_400_000), 3, (1, 2)),
    ('float32 d256 fm iq', _kw('f', 256, 'fm', True, 30000, fs=2_400_000, omega=3000), 9, (1, 2, 5)),
    ('bank 17 rows', _kw('h', 64, 'fm', False, 0, fs=2_400_000, simo=True, swap=True,
                         vfos=signals.c3_bytes(8, seed=3)[1]), 3, (2, 1)),
]


@pytest.mark.parametrize('name,kw,nch,splits', TWIN, ids=[t[0] for t in TWIN])
def test_twin_matches_seamless_oracle(name, kw, nch, splits):
    """Rotation, forward scan, fixed-horizon anticausal window, both stream boundaries, fm halo,
    SOS chaining -- the decomposition the kernels use, call by call, against the oracle."""
    pl = _plan(kw)
    body = _body(kw, nch, 5)
    ref, off = S.seamless_oracle(kw, body)
    tw = S.SeamlessTwin(pl)
    cb, outs, o, i = pl.chunk_bytes, [], 0, 0
    while o < len(body):
        k = splits[i % len(splits)]
        i += 1
        outs.append(tw.stream(body[o:o + k * cb]))
        o += k * cb
    assert abs(tw.off - off) <= 1e-12 * max(1.0, abs(off))
    outs.append(tw.end())
    out = np.concatenate(outs, axis=1)
    err = rel_err(out, ref)
    print(f'{name}: D={pl.lookahead} err={err:.2e}')
    assert out.shape == ref.shape and err < 1e-11


# max |p| and D from the design table of DESIGN.md section 11: q -> D at N = 65536/32768/16384/8192
D_TABLE = {8: (1, 1, 1, 1), 64: (1, 1, 1, 2), 256: (1, 2, 3, 6)}


@pytest.mark.parametrize('q', sorted(D_TABLE))
def test_lookahead_table_and_bound(q):
    sos = signal.cheby1(8, 0.05, 0.8 / q, output='sos')
    m = filter_modes(sos, signal.sosfilt_zi(sos))
    for N, want in zip((65536, 32768, 16384, 8192), D_TABLE[q]):
        D = lookahead_chunks(m.p, m.rho_p, N)
        assert D in (want, want + 1)
        assert lookahead_bound(m.p, m.rho_p, N, D) <= LOOKAHEAD_TOL
        assert D == 1 or lookahead_bound(m.p, m.rho_p, N, D - 1) > LOOKAHEAD_TOL


def test_seamless_plan_refusals():
    with pytest.raises(ValueError, match='divide'):
        build_plan(2_400_000, 'B', 50, [0], correct_iq=True, demod='am', omega_out=5000, seamless=True)
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    with pytest.raises(ValueError, match='smooth'):
        DspProcessor(1_024_000, dec=64, smooth=5, seamless=True)
    p = DspProcessor(1_024_000, dec=64, seamless=True)
    assert '"seamless": true' in repr(p)
    assert 'seamless' not in repr(DspProcessor(1_024_000, dec=64))
    import pickle
    assert pickle.loads(pickle.dumps(p))._seamless


def test_multigpu_refuses_seamless():
    from sdrterm_b200 import multigpu
    pl = build_plan(1_024_000, 'h', 64, [15000], demod='fm', omega_out=5000, seamless=True)
    with pytest.raises(ValueError, match='halo'):
        multigpu.TimeShardedChain(pl, max_chunks=1, device=0)
    with pytest.raises(ValueError, match='halo'):
        multigpu.RowShardedBank(1_024_000, 'h', 64, [0, 1000], max_chunks=1, device=0, seamless=True)
    with pytest.raises(ValueError, match='halo'):
        multigpu.run_file_sharded('unused', None, fs=1_024_000, enc='h', dec=64, seamless=True)


def test_cli_help_names_the_mode():
    from sdrterm_b200 import sdrterm
    ap = sdrterm.buildParser()
    assert 'not a reference option' in ap.format_help()
    a = ap.parse_args(['--seamless'])
    assert a.seamless and not ap.parse_args([]).seamless
