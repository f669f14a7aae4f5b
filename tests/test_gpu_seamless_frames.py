"""GPU: seamless streaming at any decimation (DESIGN.md section 11, frames): the plan's chunk is the
seamless frame of whole tiles (plan.seamless_frame_samples), input goes in as any number of samples
(Engine.stream_samples / sdrb_stream_samples*), and the stream's ragged end gives ceil(L/q) outputs.
Against the seamless oracles of the mode: parity, split invariance, emission accounting."""
import numpy as np
import pytest

import signals
from iq_ref import seamless_iq_oracle
from oracle import oracle as orc
from seamless_ref import _rows_use_nco, demodulate, seamless_oracle
from ssb_ref import seamless_ssb_oracle
from sdrterm_b200.plan import CHUNK_BYTES, build_plan, seamless_frame_samples
from util import rel_err

TOL = 1e-9
IQ_TOL = 1e-8
_ISZ = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'f': 4, 'd': 8}


def _kw(enc, q, demod, iq, center, fs=1_024_000, norm=False, swap=False, simo=False, vfos=None, omega=5000):
    return dict(fs=fs, enc=enc, center=center, dec=q, demod=demod, omega_out=omega, correct_iq=iq, vfos=vfos,
                simo=simo, normalize=norm, swap=swap, big_endian=None)


def _frame_plan(kw):
    ch = orc.Chain(**kw)
    sb = 2 * _ISZ[kw['enc']]
    nf = seamless_frame_samples(CHUNK_BYTES // sb, kw['dec'])
    return build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, simo=kw['simo'], swap=orc.needs_swap(ch.dt),
                      correct_iq=kw['correct_iq'], normalize=kw['normalize'], demod=kw['demod'],
                      omega_out=kw['omega_out'], seamless=True, chunk_bytes=nf * sb)


def _body(kw, nch, seed):
    n = nch * CHUNK_BYTES // (2 * _ISZ[kw['enc']])
    if kw['simo']:
        return signals.c3_bytes(n, seed=3)[0]
    return signals.generic_bytes(kw['enc'], n, seed, kw['fs'], kw['center'] or 40_000, big_endian=kw['swap'])


def _oracle(kw, body):
    if kw['demod'] == 'iq':
        return seamless_iq_oracle(kw, body)
    if kw['demod'] in ('usb', 'lsb'):
        return seamless_ssb_oracle(kw, body)
    return seamless_oracle(kw, body)


def _ragged_oracle(kw, body):
    """seamless_oracle of a stream of any whole number of samples (fm / am / re / im): decode and
    correct as the reader does over whole chunks (zero-padded), keep the stream's L samples."""
    from scipy import signal
    ch = orc.Chain(**kw)
    sb = 2 * _ISZ[kw['enc']]
    L = len(body) // sb
    st = np.frombuffer(body + bytes(-len(body) % ch.chunk_bytes), dtype=np.uint8)
    z = np.concatenate([ch.ingest(st[o:o + ch.chunk_bytes]).copy() for o in range(0, st.size, ch.chunk_bytes)])[:L]
    n = np.arange(L, dtype=np.int64)
    ys = [signal.decimate(z * np.exp(-2j * np.pi * (((int(f) * n) % kw['fs']) / kw['fs'])) if on else z, kw['dec'])
          for f, on in zip(ch.rows, _rows_use_nco(kw, ch.rows))]
    return demodulate(kw, np.array(ys))


def _iq_offset(kw, body, K):
    """The IQ corrector's offset after the stream's first K samples: off += L x_corrected per sample
    (read_file.py:65-77), so the sum of the corrected samples times L."""
    ch = orc.Chain(**kw)
    st = np.frombuffer(body + bytes(-len(body) % ch.chunk_bytes), dtype=np.uint8)
    z = np.concatenate([ch.ingest(st[o:o + ch.chunk_bytes]).copy() for o in range(0, st.size, ch.chunk_bytes)])
    return complex(np.sum(z[:K]) * (50 / kw['fs']))


def _run(eng, body, splits):
    """Feed `body` in pieces of splits[i] samples (cycled); returns the outputs, the outputs per call
    (the end call last) and the IQ offset before the end (after the whole frames)."""
    sb = eng.chunk_bytes // eng.plan.N
    outs, counts, o, i = [], [], 0, 0
    while o < len(body):
        k = splits[i % len(splits)] * sb
        i += 1
        cap = eng.stream_capacity(min(k, len(body) - o) // sb)
        r = np.asarray(eng.stream_samples(body[o:o + k]), dtype=np.float64)
        assert r.shape[1] <= cap * (eng.W // eng.M)
        counts.append(r.shape[1] // (eng.W // eng.M))
        outs.append(r)
        o += k
    iq = eng.iq_state
    cap = eng.stream_capacity(0)
    r = np.asarray(eng.stream_samples_end(), dtype=np.float64)
    assert r.shape[1] <= cap * (eng.W // eng.M)
    counts.append(r.shape[1] // (eng.W // eng.M))
    outs.append(r)
    return np.concatenate(outs, axis=1), counts, iq


CASES = [
    # BASELINE config 2: 2.4 MS/s uint8, -d 50 -w 5k, am, --correct-iq (frames of 64000 samples)
    ('config2 uint8 d50 am iq', _kw('B', 50, 'am', True, -20000, fs=2_400_000), 5),
    ('int16 d25 fm iq', _kw('h', 25, 'fm', True, 15000, fs=1_200_000), 4),
    ('int16 d3 re', _kw('h', 3, 're', False, 30000, fs=240_000), 3),
    ('int16 d5 normalize swap am', _kw('h', 5, 'am', True, 5000, norm=True, swap=True, fs=240_000), 3),
    ('float32 d100 re', _kw('f', 100, 're', False, 30000, fs=2_400_000), 4),
    ('float64 d255 im iq', _kw('d', 255, 'im', True, 12000, fs=2_400_000), 3),
    ('bank 17 rows be d50', _kw('h', 50, 'fm', False, 0, fs=2_400_000, swap=True, simo=True,
                                vfos=signals.c3_bytes(8, seed=3)[1]), 4),
    ('uint8 d50 iq', _kw('B', 50, 'iq', True, -20000, fs=2_400_000), 3),
    ('uint8 d50 usb', _kw('B', 50, 'usb', True, -20000, fs=2_400_000, omega=3000), 3),
    ('uint8 d50 lsb', _kw('B', 50, 'lsb', False, 20000, fs=2_400_000, omega=3000), 3),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,kw,nch', CASES, ids=[c[0] for c in CASES])
def test_frames_match_oracle(name, kw, nch):
    from sdrterm_b200.engine import Engine
    pl = _frame_plan(kw)
    body = _body(kw, nch, 200 + pl.q)
    ref, off = _oracle(kw, body)
    L = len(body) // (pl.chunk_bytes // pl.N)
    ncn = CHUNK_BYTES // (pl.chunk_bytes // pl.N)        # reader chunk in samples
    off = _iq_offset(kw, body, L // pl.N * pl.N) if kw['correct_iq'] else 0j
    res, iqs = [], []
    with Engine(pl, max_chunks=4) as eng:
        for splits in ((ncn,), (2 * ncn,), (3 * ncn,), (1, 7, 4097, 12345, 70001)):
            out, counts, iq = _run(eng, body, splits)
            assert out.shape == ref.shape and out.shape[1] == -(-L // pl.q) * (pl.W // pl.M)
            # each call but the end emits whole frames: its final frames times M
            assert all(c % pl.M == 0 for c in counts[:-1])
            iqs.append(iq)
            res.append(out)
    err = rel_err(res[0], ref)
    spread = max(rel_err(o, res[0]) for o in res[1:])
    iq_err = max(abs(v - off) for v in iqs) / max(1.0, abs(off))
    bad = np.argwhere(np.abs(res[0] - ref) > 1e-9 * max(1.0, np.max(np.abs(ref))))
    print(f'{name}: N_f={pl.N} M_f={pl.M} D={pl.lookahead} L={L} Lp={L % pl.N} err={err:.3e} spread={spread:.3e} '
          f'iq={iq_err:.3e} bad={len(bad)} first={bad[:3].tolist()} width={ref.shape[1]}')
    assert err < TOL
    if kw['correct_iq']:
        assert iq_err <= IQ_TOL
    assert spread <= 1e-12


@pytest.mark.gpu
def test_frames_accounting():
    """Per call: max(0, frames seen - D) - frames emitted, times M_f; the end emits the rest."""
    from sdrterm_b200.engine import Engine
    kw = _kw('B', 50, 'am', True, -20000, fs=2_400_000)
    pl = _frame_plan(kw)
    body = _body(kw, 6, 5)
    sb = pl.chunk_bytes // pl.N
    L = len(body) // sb
    with Engine(pl, max_chunks=4) as eng:
        D = eng.lookahead
        split = 50_000
        out, counts, _ = _run(eng, body, (split,))
    seen_s, emitted = 0, 0
    for c in counts[:-1]:
        seen_s = min(L, seen_s + split)
        final = max(0, seen_s // pl.N - D)
        assert c == (final - emitted) * pl.M
        emitted = final
    assert sum(counts) == -(-L // pl.q)


@pytest.mark.gpu
@pytest.mark.parametrize('kw', [_kw('h', 64, 'fm', True, 15000), _kw('B', 8, 'iq', True, -20000, fs=2_400_000)],
                         ids=['int16-d64-fm', 'uint8-d8-iq'])
def test_power_of_two_samples_equal_chunks(kw):
    """Power-of-two q: frames are the chunks; the sample entries on whole chunks are bit-identical."""
    from sdrterm_b200.engine import Engine
    pl = _frame_plan(kw)
    assert pl.N * (pl.chunk_bytes // pl.N) == CHUNK_BYTES
    body = _body(kw, 2 * (pl.lookahead + 1) + 1, 9)
    with Engine(pl, max_chunks=4) as eng:
        a = [eng.stream(body[:2 * CHUNK_BYTES]), eng.stream(body[2 * CHUNK_BYTES:]), eng.stream_end()]
        b = [eng.stream_samples(body[:2 * CHUNK_BYTES]), eng.stream_samples(body[2 * CHUNK_BYTES:]),
             eng.stream_samples_end()]
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x), np.asarray(y))


@pytest.mark.gpu
def test_long_stream_d50():
    """300 reader chunks at -d 50 through many calls."""
    from sdrterm_b200.engine import Engine
    kw = _kw('B', 50, 'am', True, -20000, fs=2_400_000)
    pl = _frame_plan(kw)
    body = _body(kw, 300, 8)
    ref, _ = seamless_oracle(kw, body)
    L = len(body) // 2
    off = _iq_offset(kw, body, L // pl.N * pl.N)
    with Engine(pl, max_chunks=64) as eng:
        out, _, iq = _run(eng, body, (64 * 65536, 17 * 65536 + 3, 1, 40 * 65536 - 1))
    err = rel_err(out, ref)
    print(f'300 chunks d50: err={err:.3e} iq={abs(iq - off) / abs(off):.3e}')
    assert out.shape == ref.shape and err < TOL
    assert abs(iq - off) <= IQ_TOL * max(1.0, abs(off))


@pytest.mark.gpu
def test_refusals_and_pending_state():
    from sdrterm_b200 import _native as nat
    from sdrterm_b200.engine import Engine
    kw = _kw('B', 50, 'am', False, 0, fs=2_400_000)
    pl = _frame_plan(kw)
    body = _body(kw, 1, 3)
    with Engine(pl, max_chunks=2) as eng:
        assert eng.stream_samples(body[:2 * 27]).shape == (1, 0)
        with pytest.raises(nat.SdrbError):
            eng.stream_samples_end()                  # 27 samples: scipy refuses it too
        eng.stream_samples(body[:2 * 1000])
        with pytest.raises(nat.SdrbError):
            eng.stream_end()                          # a partial frame is pending
        with pytest.raises(nat.SdrbError):
            eng.stream(body[:pl.chunk_bytes])
        out = eng.stream_samples_end()
        ref = _ragged_oracle(kw, body[:2 * 1000])    # head and end in one partial frame
        assert out.shape == ref.shape and rel_err(out, ref) < TOL
        # one input kind per stream: chunks, then samples (or the reverse) is refused until the end
        eng.stream(body[:pl.chunk_bytes])
        with pytest.raises(nat.SdrbError):
            eng.stream_samples(body[:2 * 10])
        eng.stream_end()
        eng.stream_samples(body[:2 * 10])
        with pytest.raises(nat.SdrbError):
            eng.stream(body[:pl.chunk_bytes])
        with pytest.raises(nat.SdrbError):
            eng.stream_samples_end()                  # 10 samples: refused, and the stream is reset
        assert eng.stream(body[:pl.chunk_bytes]).shape[1] == 0


@pytest.mark.gpu
def test_fm_single_output_refused():
    """fm of a stream of at most q samples has one output and no discriminator pair: refused."""
    from sdrterm_b200 import _native as nat
    from sdrterm_b200.engine import Engine
    kw = _kw('B', 50, 'fm', False, 0, fs=2_400_000)
    pl = _frame_plan(kw)
    body = _body(kw, 1, 3)
    with Engine(pl, max_chunks=2) as eng:
        eng.stream_samples(body[:2 * 50])
        with pytest.raises(nat.SdrbError):
            eng.stream_samples_end()
        eng.stream_samples(body[:2 * 51])
        ref = _ragged_oracle(kw, body[:2 * 51])
        out = eng.stream_samples_end()
        assert out.shape == ref.shape == (1, 2) and rel_err(out, ref) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize('Lp', [10, 27, 28, 49, 50, 51])
def test_short_ragged_end(Lp):
    """A ragged last frame shorter than the pad (its end window reaches into the frame before) and
    around one block."""
    from sdrterm_b200.engine import Engine
    kw = _kw('B', 50, 'am', True, -20000, fs=2_400_000)
    pl = _frame_plan(kw)
    body = _body(kw, 3, 4)[:2 * (2 * pl.N + Lp)]
    ref = _ragged_oracle(kw, body)
    with Engine(pl, max_chunks=4) as eng:
        out, _, _ = _run(eng, body, (7001,))
    err = rel_err(out, ref)
    print(f'Lp={Lp}: err={err:.3e}')
    assert out.shape == ref.shape and err < TOL


@pytest.mark.gpu
@pytest.mark.parametrize('demod', ['am', 'fm'])
def test_no_transient_at_frame_edges(demod):
    """A steady carrier (am) or tone (fm) at -d 50: the seamless output follows the oracle's smooth
    value across every frame and chunk edge."""
    from sdrterm_b200.engine import Engine
    fs, q = 2_400_000, 50
    kw = _kw('B', q, demod, False, 0, fs=fs)
    pl = _frame_plan(kw)
    n = 5 * CHUNK_BYTES // 2
    t = np.arange(n)
    x = 0.8 * np.exp(2j * np.pi * (3000 * t / fs if demod == 'fm' else 0.0) + 0.3j)
    raw = np.empty(2 * n, dtype=np.uint8)
    raw[0::2] = np.clip(np.round(127.5 + 127 * x.real), 0, 255)
    raw[1::2] = np.clip(np.round(127.5 + 127 * x.imag), 0, 255)
    body = raw.tobytes()
    ref, _ = seamless_oracle(kw, body)
    with Engine(pl, max_chunks=4) as eng:
        out, _, _ = _run(eng, body, (4097,))
    edges = [e // q for e in list(range(pl.N, n, pl.N)) + list(range(CHUNK_BYTES // 2, n, CHUNK_BYTES // 2))]
    dev = max(np.max(np.abs(out[:, e - 3:e + 3] - ref[:, e - 3:e + 3])) for e in edges)
    print(f'{demod}: max deviation from the oracle around {len(edges)} frame / chunk edges: {dev:.3e}')
    assert dev < 1e-9 * max(1.0, np.max(np.abs(ref)))


def _cli_env():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return dict(os.environ, PYTHONPATH=os.path.join(root, 'src'))


@pytest.mark.gpu
def test_cli_config2_raw_matches_oracle(tmp_path):
    """`python -m sdrterm -e B -r 2400k -d 50 -m am --correct-iq --seamless` on a raw file: 48 kHz
    click-free audio, the ragged end included."""
    import subprocess
    import sys
    kw = _kw('B', 50, 'am', True, 0, fs=2_400_000)
    body = _body(kw, 5, 21)
    fin, fout = tmp_path / 'in.raw', tmp_path / 'out.bin'
    fin.write_bytes(body)
    subprocess.run([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-o', str(fout), '-e', 'B', '-r', '2400k',
                    '-d', '50', '-w', '5k', '-m', 'am', '--correct-iq', '--seamless'], env=_cli_env(), cwd=str(tmp_path),
                   check=True, timeout=300, capture_output=True)
    ref, _ = seamless_oracle(kw, body)
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')[None]
    err = rel_err(got, ref)
    print(f'CLI -d 50 --seamless: outputs={got.shape[1]} err={err:.3e}')
    assert got.shape == ref.shape and err < TOL


@pytest.mark.gpu
def test_cli_simo_d50_sockets_match_oracle(tmp_path):
    """`--simo --seamless -d 50`: one big-endian stream per VFO socket, each the oracle's row."""
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
    proc = subprocess.Popen([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-r', '2400k', '-e', 'h', '-X', '-d', '50',
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
    kw = _kw('h', 50, 'fm', False, 0, fs=2_400_000, swap=True, simo=True, vfos=vf)
    ref, _ = seamless_oracle(kw, body)
    rows = [np.frombuffer(got[i][:len(got[i]) // 8 * 8], dtype='>f8').astype(np.float64) for i in range(3)]
    assert all(g.shape == ref[0].shape for g in rows)
    # sockets are not tied to rows in connection order: each stream matches one row, all rows covered
    match = [int(np.argmin([rel_err(g, r) for r in ref])) for g in rows]
    errs = [rel_err(g, ref[j]) for g, j in zip(rows, match)]
    print(f'CLI --simo -d 50 --seamless: outputs={[g.size for g in rows]} rows={match} err={max(errs):.3e}')
    assert sorted(match) == list(range(len(ref))) and max(errs) < TOL
