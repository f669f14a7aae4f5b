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


@pytest.mark.gpu
def test_seamless_refuses_chunk_local_entry_points():
    from sdrterm_b200 import _native as nat
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, 'fm', True, 15000)
    pl = _plan(kw)
    with Engine(pl, max_chunks=2) as eng:
        with pytest.raises(nat.SdrbError):
            eng.process(_body(kw, 1, 1))
        with pytest.raises(ValueError):
            eng.set_smooth(5)
        rc = nat.lib().sdrb_set_smooth(eng._h, 5, 2, 2, -2, np.zeros(25).ctypes.data)
        assert rc == -1
        rc = nat.lib().sdrb_iq_gain(eng._h, _body(kw, 1, 1), 1)
        assert rc == -4


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
