"""GPU: the seamless streaming mode (Engine.stream / stream_end, DESIGN.md section 11) against the
seamless oracle of tests/seamless_ref.py: parity, batch invariance, emission accounting, and what
the mode is for -- no transient at chunk edges."""
import numpy as np
import pytest

import signals
from oracle import oracle as orc
from seamless_ref import seamless_oracle
from sdrterm_b200.plan import build_plan
from util import rel_err

TOL = 1e-9
# the IQ offset after a stream of int16 chunks on k_tc: its tile aggregates come out of the
# fixed-point GEMM, ~1e-9 relative after a few chunks (observed 1.2e-9); the outputs stay ~5e-12
IQ_TOL = 1e-8
_ISZ = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'f': 4, 'd': 8}


def _kw(enc, q, demod, iq, center, fs=1_024_000, norm=False, swap=False, simo=False, vfos=None, omega=5000):
    return dict(fs=fs, enc=enc, center=center, dec=q, demod=demod, omega_out=omega, correct_iq=iq, vfos=vfos,
                simo=simo, normalize=norm, swap=swap, big_endian=None)


def _plan(kw):
    ch = orc.Chain(**kw)
    return build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, simo=kw['simo'], swap=orc.needs_swap(ch.dt),
                      correct_iq=kw['correct_iq'], normalize=kw['normalize'], demod=kw['demod'],
                      omega_out=kw['omega_out'], seamless=True)


def _body(kw, nch, seed):
    n = nch * 131072 // (2 * _ISZ[kw['enc']])
    if kw['simo']:        # a carrier in every VFO of the bank (config 3's signal)
        return signals.c3_bytes(n, seed=3)[0]
    return signals.generic_bytes(kw['enc'], n, seed, kw['fs'], kw['center'] or 40_000, big_endian=kw['swap'])


def _run(eng, body, splits):
    cb = eng.chunk_bytes
    outs, o, i, counts = [], 0, 0, []
    while o < len(body):
        k = splits[i % len(splits)]
        i += 1
        r = eng.stream(body[o:o + k * cb])
        counts.append(r.shape[1] // eng.M)
        outs.append(np.asarray(r, dtype=np.float64))
        o += k * cb
    iq = eng.iq_state
    outs.append(np.asarray(eng.stream_end(), dtype=np.float64))
    return np.concatenate(outs, axis=1), counts, iq


CASES = [
    ('int16 d64 fm iq k_tc', _kw('h', 64, 'fm', True, 15000), True, None),
    ('int16 d64 fm iq k_main', _kw('h', 64, 'fm', True, 15000), False, None),
    ('int16 d64 am centre0', _kw('h', 64, 'am', False, 0), True, None),
    ('uint8 d8 am iq', _kw('B', 8, 'am', True, -20000, fs=2_400_000), True, None),
    ('float32 d256 re', _kw('f', 256, 're', False, 30000, fs=2_400_000), True, None),
    ('float64 d32 im iq', _kw('d', 32, 'im', True, 12000, fs=192_000), True, None),
    ('int16 normalize swap am iq', _kw('h', 16, 'am', True, 5000, norm=True, swap=True, fs=500_000), True, None),
    ('int16 bank 17 rows be', _kw('h', 64, 'fm', False, 0, fs=2_400_000, swap=True, simo=True,
                                  vfos=signals.c3_bytes(8, seed=3)[1]), True, 'c3'),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,kw,use_tc,_', CASES, ids=[c[0] for c in CASES])
def test_seamless_matches_oracle(name, kw, use_tc, _):
    from sdrterm_b200.engine import Engine
    pl = _plan(kw)
    nch = 3 * (pl.lookahead + 1)
    body = _body(kw, nch, 100 + pl.q)
    ref, off = seamless_oracle(kw, body)
    with Engine(pl, max_chunks=4, use_tc=use_tc) as eng:
        out, counts, iq = _run(eng, body, (1, 2, 3))
    err = rel_err(out, ref)
    print(f'{name}: D={pl.lookahead} chunks={nch} rows={pl.R} err={err:.3e}')
    assert out.shape == ref.shape and err < TOL
    if kw['correct_iq']:
        assert abs(iq - off) <= IQ_TOL * max(1.0, abs(off))


@pytest.mark.gpu
def test_seamless_long_stream():
    """300 chunks through many calls: the forward state, the SOS state and the window carried on."""
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, 'fm', True, 15000)
    pl = _plan(kw)
    body = _body(kw, 300, 7)
    ref, off = seamless_oracle(kw, body)
    with Engine(pl, max_chunks=64) as eng:
        out, counts, iq = _run(eng, body, (64, 17, 1, 40))
    err = rel_err(out, ref)
    print(f'300 chunks: err={err:.3e}')
    assert out.shape == ref.shape and err < TOL
    assert abs(iq - off) <= IQ_TOL * max(1.0, abs(off))


@pytest.mark.gpu
@pytest.mark.parametrize('kw', [_kw('h', 64, 'am', True, 15000), _kw('f', 256, 'fm', True, 30000, fs=2_400_000, omega=3000)],
                         ids=['int16-d64', 'float32-d256'])
def test_seamless_batch_invariance_and_accounting(kw):
    from sdrterm_b200.engine import Engine
    pl = _plan(kw)
    D = pl.lookahead
    nch = 3 * (D + 1) + 2
    body = _body(kw, nch, 11)
    ref, off = seamless_oracle(kw, body)
    res = []
    with Engine(pl, max_chunks=8) as eng:
        assert eng.lookahead == D
        for split in (1, 2, 5, 8):
            out, counts, iq = _run(eng, body, (split,))
            seen, emitted = 0, 0
            for k in counts:                       # per call: max(0, seen - D) - emitted chunks
                seen = min(nch, seen + split)
                assert k == max(0, seen - D) - emitted
                emitted += k
            assert out.shape[1] == nch * pl.M     # stream_end emitted the rest
            assert abs(iq - off) <= IQ_TOL * max(1.0, abs(off))
            res.append(out)
    for o in res[1:]:
        assert rel_err(o, res[0]) <= 1e-12
    assert rel_err(res[0], ref) < TOL


@pytest.mark.gpu
def test_seamless_short_and_empty_streams():
    from sdrterm_b200.engine import Engine
    kw = _kw('f', 256, 'am', False, 30000, fs=2_400_000, omega=3000)
    pl = _plan(kw)
    assert pl.lookahead >= 2
    with Engine(pl, max_chunks=4) as eng:
        assert eng.stream_end().shape == (1, 0)                   # empty stream
        body = _body(kw, pl.lookahead - 1, 3)                     # shorter than D
        first = eng.stream(body)
        assert first.shape == (1, 0)
        out = eng.stream_end()
        ref, _ = seamless_oracle(kw, body)
        assert out.shape == ref.shape and rel_err(out, ref) < TOL
        body2 = _body(kw, pl.lookahead + 2, 4)                    # a second stream after stream_end
        out2 = np.concatenate([eng.stream(body2), eng.stream_end()], axis=1)
        ref2, _ = seamless_oracle(kw, body2)
        assert rel_err(out2, ref2) < TOL


OK, ARG, STATE = 0, -1, -4     # SDRB_OK, SDRB_ERR_ARG, SDRB_ERR_STATE
MAXC = 2                       # max_chunks of the handles below
# Misuse of every handle entry point, called through the C ABI on a chunk-local handle and on a
# seamless one: (case, demod, call, code on the chunk-local handle, code on the seamless handle).
# `call(L, h, b)` gets the library, the handle and the buffers of _misuse_buffers; fm handles run
# the IQ corrector, iq handles do not.  Zero chunks: sdrb_submit refuses them, the other
# chunk-local calls are a successful no-op, the stream calls run.
MISUSE = [
    # null pointers (a null handle is refused first, whatever the call)
    ('process_device null handle', 'fm', lambda L, h, b: L.sdrb_process_device(None, b.raw_d, 1, b.out_d, None), ARG, ARG),
    ('process_device null raw', 'fm', lambda L, h, b: L.sdrb_process_device(h, None, 1, b.out_d, None), ARG, ARG),
    ('process_device null out', 'fm', lambda L, h, b: L.sdrb_process_device(h, b.raw_d, 1, None, None), ARG, ARG),
    ('submit null handle', 'fm', lambda L, h, b: L.sdrb_submit(None, 0, b.raw_h, 1, b.out_h), ARG, ARG),
    ('submit null raw', 'fm', lambda L, h, b: L.sdrb_submit(h, 0, None, 1, b.out_h), ARG, ARG),
    ('submit null out', 'fm', lambda L, h, b: L.sdrb_submit(h, 0, b.raw_h, 1, None), ARG, ARG),
    ('process null handle', 'fm', lambda L, h, b: L.sdrb_process(None, b.raw_h, 1, b.out_h), ARG, ARG),
    ('process null raw', 'fm', lambda L, h, b: L.sdrb_process(h, None, 1, b.out_h), ARG, ARG),
    ('process null out', 'fm', lambda L, h, b: L.sdrb_process(h, b.raw_h, 1, None), ARG, ARG),
    ('process null buffers 0 chunks', 'fm', lambda L, h, b: L.sdrb_process(h, None, 0, None), OK, STATE),
    ('stream_device null handle', 'fm', lambda L, h, b: L.sdrb_stream_device(None, b.raw_d, 1, b.out_d, None, b.got), ARG, ARG),
    ('stream_device null raw', 'fm', lambda L, h, b: L.sdrb_stream_device(h, None, 1, b.out_d, None, b.got), ARG, ARG),
    ('stream_device null raw 0 chunks', 'fm', lambda L, h, b: L.sdrb_stream_device(h, None, 0, b.out_d, None, b.got), STATE, OK),
    ('stream_device null out', 'fm', lambda L, h, b: L.sdrb_stream_device(h, b.raw_d, 1, None, None, b.got), ARG, ARG),
    ('stream_end_device null handle', 'fm', lambda L, h, b: L.sdrb_stream_end_device(None, b.out_d, None, b.got), ARG, ARG),
    ('stream_end_device null out', 'fm', lambda L, h, b: L.sdrb_stream_end_device(h, None, None, b.got), ARG, ARG),
    ('stream null handle', 'fm', lambda L, h, b: L.sdrb_stream(None, b.raw_h, 1, b.out_h, b.got), ARG, ARG),
    ('stream null raw', 'fm', lambda L, h, b: L.sdrb_stream(h, None, 1, b.out_h, b.got), ARG, ARG),
    ('stream null out', 'fm', lambda L, h, b: L.sdrb_stream(h, b.raw_h, 1, None, b.got), ARG, ARG),
    ('stream_end null handle', 'fm', lambda L, h, b: L.sdrb_stream_end(None, b.out_h, b.got), ARG, ARG),
    ('stream_end null out', 'fm', lambda L, h, b: L.sdrb_stream_end(h, None, b.got), ARG, ARG),
    ('iq_gain null handle', 'fm', lambda L, h, b: L.sdrb_iq_gain(None, b.raw_h, 1), ARG, ARG),
    ('iq_gain null raw', 'fm', lambda L, h, b: L.sdrb_iq_gain(h, None, 1), ARG, ARG),
    ('phases null handle', 'fm', lambda L, h, b: L.sdrb_process_device_phases(None, b.raw_d, 1, b.out_d, None, 7), ARG, ARG),
    ('phases null raw', 'fm', lambda L, h, b: L.sdrb_process_device_phases(h, None, 1, b.out_d, None, 7), ARG, ARG),
    ('phases null out with finish', 'fm', lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, 1, None, None, 7), ARG, ARG),
    ('phases null out without finish', 'fm', lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, 1, None, None, 3), OK, STATE),
    ('iq_export null handle', 'fm', lambda L, h, b: L.sdrb_iq_export_device(None, b.g3_d, 1.0, None), ARG, ARG),
    ('iq_export null dst', 'fm', lambda L, h, b: L.sdrb_iq_export_device(h, None, 1.0, None), ARG, ARG),
    ('iq_prefix null handle', 'fm', lambda L, h, b: L.sdrb_iq_prefix_device(None, b.g3_d, 0, None), ARG, ARG),
    ('iq_prefix null gains', 'fm', lambda L, h, b: L.sdrb_iq_prefix_device(h, None, 0, None), ARG, ARG),
    ('iq_prefix rank -1', 'fm', lambda L, h, b: L.sdrb_iq_prefix_device(h, b.g3_d, -1, None), ARG, ARG),
    # zero chunks
    ('process_device 0 chunks', 'fm', lambda L, h, b: L.sdrb_process_device(h, b.raw_d, 0, b.out_d, None), OK, STATE),
    ('submit 0 chunks', 'fm', lambda L, h, b: L.sdrb_submit(h, 0, b.raw_h, 0, b.out_h), ARG, STATE),
    ('process 0 chunks', 'fm', lambda L, h, b: L.sdrb_process(h, b.raw_h, 0, b.out_h), OK, STATE),
    ('stream_device 0 chunks', 'fm', lambda L, h, b: L.sdrb_stream_device(h, b.raw_d, 0, b.out_d, None, b.got), STATE, OK),
    ('stream 0 chunks', 'fm', lambda L, h, b: L.sdrb_stream(h, b.raw_h, 0, b.out_h, b.got), STATE, OK),
    ('iq_gain 0 chunks', 'fm', lambda L, h, b: L.sdrb_iq_gain(h, b.raw_h, 0), OK, STATE),
    ('phases 0 chunks', 'fm', lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, 0, b.out_d, None, 7), OK, STATE),
    # max_chunks + 1 (sdrb_process takes any number: it runs them in batches)
    ('process_device max+1', 'fm', lambda L, h, b: L.sdrb_process_device(h, b.raw_d, MAXC + 1, b.out_d, None), ARG, STATE),
    ('submit max+1', 'fm', lambda L, h, b: L.sdrb_submit(h, 0, b.raw_h, MAXC + 1, b.out_h), ARG, STATE),
    ('process max+1', 'fm', lambda L, h, b: L.sdrb_process(h, b.raw_h, MAXC + 1, b.out_h), OK, STATE),
    ('stream_device max+1', 'fm', lambda L, h, b: L.sdrb_stream_device(h, b.raw_d, MAXC + 1, b.out_d, None, b.got), STATE, ARG),
    ('stream max+1', 'fm', lambda L, h, b: L.sdrb_stream(h, b.raw_h, MAXC + 1, b.out_h, b.got), STATE, ARG),
    ('iq_gain max+1', 'fm', lambda L, h, b: L.sdrb_iq_gain(h, b.raw_h, MAXC + 1), ARG, STATE),
    ('iq_gain max+1 without corrector', 'iq', lambda L, h, b: L.sdrb_iq_gain(h, b.raw_h, MAXC + 1), OK, STATE),
    ('phases max+1', 'fm', lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, MAXC + 1, b.out_d, None, 7), ARG, STATE),
    # the wrong kind of handle for a valid call
    ('process_device', 'fm', lambda L, h, b: L.sdrb_process_device(h, b.raw_d, 1, b.out_d, None), OK, STATE),
    ('submit + wait', 'fm', lambda L, h, b: L.sdrb_submit(h, 1, b.raw_h, 1, b.out_h) or L.sdrb_wait(h, 1), OK, STATE),
    ('process', 'fm', lambda L, h, b: L.sdrb_process(h, b.raw_h, 1, b.out_h), OK, STATE),
    ('stream_device', 'fm', lambda L, h, b: L.sdrb_stream_device(h, b.raw_d, 1, b.out_d, None, b.got), STATE, OK),
    ('stream_end_device', 'fm', lambda L, h, b: L.sdrb_stream_end_device(h, b.out_d, None, b.got), STATE, OK),
    ('stream', 'fm', lambda L, h, b: L.sdrb_stream(h, b.raw_h, 1, b.out_h, b.got), STATE, OK),
    ('stream_end', 'fm', lambda L, h, b: L.sdrb_stream_end(h, b.out_h, b.got), STATE, OK),
    ('iq_gain', 'fm', lambda L, h, b: L.sdrb_iq_gain(h, b.raw_h, 1), OK, STATE),
    ('phases', 'fm', lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, 1, b.out_d, None, 7), OK, STATE),
    ('iq_export', 'fm', lambda L, h, b: L.sdrb_iq_export_device(h, b.g3_d, 1.0, None), OK, STATE),
    ('iq_prefix', 'fm', lambda L, h, b: L.sdrb_iq_prefix_device(h, b.g3_d, 0, None), OK, STATE),
    ('set_smooth', 'fm', lambda L, h, b: L.sdrb_set_smooth(h, 5, 2, 2, -2, b.smooth), OK, ARG),
    # slots
    ('submit slot -1', 'fm', lambda L, h, b: L.sdrb_submit(h, -1, b.raw_h, 1, b.out_h), ARG, ARG),
    ('submit slot 2', 'fm', lambda L, h, b: L.sdrb_submit(h, 2, b.raw_h, 1, b.out_h), ARG, ARG),
    ('wait slot -1', 'fm', lambda L, h, b: L.sdrb_wait(h, -1), ARG, ARG),
    ('wait slot 2', 'fm', lambda L, h, b: L.sdrb_wait(h, 2), ARG, ARG),
    # device outputs 8 bytes off: iq stores 16-byte (Re, Im) pairs, real rows 8-byte doubles
    ('process_device out+8 iq', 'iq', lambda L, h, b: L.sdrb_process_device(h, b.raw_d, 1, b.out_d + 8, None), ARG, STATE),
    ('process_device out+8 fm', 'fm', lambda L, h, b: L.sdrb_process_device(h, b.raw_d, 1, b.out_d + 8, None), OK, STATE),
    ('phases out+8 iq', 'iq', lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, 1, b.out_d + 8, None, 7), ARG, STATE),
    ('phases out+8 iq without finish', 'iq',
     lambda L, h, b: L.sdrb_process_device_phases(h, b.raw_d, 1, b.out_d + 8, None, 3), OK, STATE),
    ('stream_device out+8 iq', 'iq', lambda L, h, b: L.sdrb_stream_device(h, b.raw_d, 1, b.out_d + 8, None, b.got), STATE, ARG),
    ('stream_device out+8 fm', 'fm', lambda L, h, b: L.sdrb_stream_device(h, b.raw_d, 1, b.out_d + 8, None, b.got), STATE, OK),
    ('stream_end_device out+8 iq', 'iq', lambda L, h, b: L.sdrb_stream_end_device(h, b.out_d + 8, None, b.got), STATE, ARG),
]


def _misuse_buffers(kw, eng):
    import ctypes as C
    import torch
    from types import SimpleNamespace
    nout = (MAXC + 1 + eng.lookahead + 2) * eng.R * eng.W       # rows of any call above, plus slack for +8
    raw = np.frombuffer(_body(kw, MAXC + 1, 1), dtype=np.uint8).copy()
    b = SimpleNamespace(raw=raw, raw_dt=torch.from_numpy(raw).cuda(), out_dt=torch.zeros(nout, dtype=torch.float64, device='cuda'),
                        g3=torch.zeros(6, dtype=torch.float64, device='cuda'), out=np.zeros(nout), sm=np.zeros(25),
                        got=C.pointer(C.c_size_t(0)))
    b.raw_h, b.out_h, b.smooth = b.raw.ctypes.data, b.out.ctypes.data, b.sm.ctypes.data
    b.raw_d, b.out_d, b.g3_d = b.raw_dt.data_ptr(), b.out_dt.data_ptr(), b.g3.data_ptr()
    return b


@pytest.mark.gpu
def test_entry_points_refuse_misuse():
    """Every handle entry point returns the same code for the same misuse, on both kinds of handle."""
    import torch
    from sdrterm_b200 import _native as nat
    from sdrterm_b200.engine import Engine
    L = nat.lib()
    got = []
    for demod, iq in (('fm', True), ('iq', False)):
        kw = _kw('h', 64, demod, iq, 15000)
        for col in (3, 4):
            pl = build_plan(kw['fs'], 'h', 64, [15000], correct_iq=iq, demod=demod, omega_out=5000, seamless=col == 4)
            with Engine(pl, max_chunks=MAXC) as eng:
                b = _misuse_buffers(kw, eng)
                for case in MISUSE:
                    if case[1] == demod:
                        rc = case[2](L, eng._h, b)
                        torch.cuda.synchronize()
                        got.append((case[0], 'seamless' if col == 4 else 'chunk-local', rc, case[col]))
                if col == 4:
                    with pytest.raises(nat.SdrbError):
                        eng.process(_body(kw, 1, 1))
                    with pytest.raises(ValueError):
                        eng.set_smooth(5)
    bad = [g for g in got if g[2] != g[3]]
    assert not bad, bad
    assert len(got) == 2 * len(MISUSE)


def _edge_error(out, ref, M, halfwidth=8):
    """Largest relative deviation within +-halfwidth outputs of every chunk edge (steady part only)."""
    idx = np.concatenate([np.arange(c * M - halfwidth, c * M + halfwidth) for c in range(1, out.shape[1] // M)])
    return float(np.max(np.abs(out[:, idx] - ref[:, idx])) / np.max(np.abs(ref)))


@pytest.mark.gpu
@pytest.mark.parametrize('demod', ['am', 'fm'])
def test_no_transient_at_chunk_edges(demod):
    """A steady AM carrier / an FM tone: the seamless output is the oracle's smooth value across every
    chunk edge, while the default engine on the same input still shows its per-chunk transient."""
    from sdrterm_b200.engine import Engine
    fs, center, nch = 1_024_000, 15000, 6
    n = nch * 32768
    t = np.arange(n)
    if demod == 'am':
        x = 0.5 * np.exp(2j * np.pi * center * t / fs)
    else:
        x = 0.5 * np.exp(2j * np.pi * (center * t / fs + 3.0 * np.sin(2 * np.pi * 700 * t / fs)))
    iq = np.empty(2 * n, dtype='<i2')
    iq[0::2] = np.round(20000 * x.real)
    iq[1::2] = np.round(20000 * x.imag)
    body = iq.tobytes()
    kw = _kw('h', 64, demod, False, center)
    ref, _ = seamless_oracle(kw, body)
    pl = _plan(kw)
    with Engine(pl, max_chunks=nch) as eng:
        out = np.concatenate([eng.stream(body), eng.stream_end()], axis=1)
    M = pl.M
    err = _edge_error(out, ref, M)
    print(f'{demod}: seamless edge error {err:.3e}')
    assert err < TOL
    pld = build_plan(fs, 'h', 64, [center], demod=demod, omega_out=5000)
    with Engine(pld, max_chunks=nch) as eng:
        dflt = eng.process(body)
    assert rel_err(dflt, orc.Chain(**kw).run(body)) < TOL          # the default output is unchanged
    derr = _edge_error(dflt, ref, M)
    print(f'{demod}: default edge deviation {derr:.3e}')
    assert derr > 1e-4


def _cli_env():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return dict(os.environ, PYTHONPATH=os.path.join(root, 'src'))


@pytest.mark.gpu
def test_cli_seamless_wav_matches_oracle(tmp_path):
    """`python -m sdrterm --seamless` with config 1's flags on a WAV file (dataOffset and stale-tail
    quirks of the reader included)."""
    import subprocess
    import sys
    from util import parse_wav
    raw = signals.c1_bytes(4 * 32768 + 5000, seed=0)
    fin, fout = tmp_path / 'in.wav', tmp_path / 'out.bin'
    fin.write_bytes(raw)
    subprocess.run([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-o', str(fout), '-c', '15000', '-w', '5000',
                    '-d', '64', '-m', 'fm', '--correct-iq', '--seamless'], env=_cli_env(), cwd=str(tmp_path),
                   check=True, timeout=300, capture_output=True)
    fs, enc, be, off = parse_wav(raw)
    kw = _kw(enc, 64, 'fm', True, 15000, fs=fs)
    ref, _ = seamless_oracle(kw, raw[off:])
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')[None]
    err = rel_err(got, ref)
    print(f'CLI --seamless: err={err:.3e}')
    assert got.shape == ref.shape and err < TOL


@pytest.mark.gpu
def test_cli_simo_seamless_sockets_match_oracle(tmp_path):
    """`--simo --seamless`: one big-endian stream per VFO socket, each the seamless oracle's row."""
    import socket
    import subprocess
    import sys
    import threading
    import time
    body, vfos = signals.c3_bytes(4 * 32768, seed=3)
    vf = ','.join(vfos.split(',')[:2])
    fin = tmp_path / 'in.raw'
    fin.write_bytes(body)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    proc = subprocess.Popen([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-r', '2400k', '-e', 'h', '-X', '-d', '64',
                             '-w', '5k', '--simo', f'--vfos={vf}', '--vfo-host', f'127.0.0.1:{port}', '--seamless'],
                            env=_cli_env(), cwd=str(tmp_path), stderr=subprocess.PIPE, text=True)
    head = ''
    deadline = time.time() + 120
    while time.time() < deadline and 'Accepting' not in head:
        line = proc.stderr.readline()
        if not line:
            break
        head += line
    assert '"seamless": true' in head, head
    got = {}

    def client(i):
        c = socket.create_connection(('127.0.0.1', port), timeout=30)
        buf = b''
        while True:
            d = c.recv(1 << 16)
            if not d:
                break
            buf += d
        got[i] = buf
        c.close()

    cl = [threading.Thread(target=client, args=(i,), daemon=True) for i in range(3)]
    for t in cl:
        t.start()
    proc.stderr.read()
    proc.wait(120)
    for t in cl:
        t.join(30)
    kw = _kw('h', 64, 'fm', False, 0, fs=2_400_000, swap=True, simo=True, vfos=vf)
    ref, _ = seamless_oracle(kw, body)
    # sockets are not tied to rows in connection order: match each received stream to its row
    got_rows = [np.frombuffer(got[i][:len(got[i]) // 8 * 8], dtype='>f8').astype(np.float64) for i in range(3)]
    for g in got_rows:
        assert g.shape == ref[0].shape
        assert min(rel_err(g, r) for r in ref) < TOL
