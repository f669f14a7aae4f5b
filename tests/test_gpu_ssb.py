"""GPU: single-sideband output (``-m usb`` / ``-m lsb``) against its oracle (tests/ssb_ref.py) through
every layer: the fused k_finish, the general k_fixup + k_demod path, the seamless mode, the banks,
submit/wait, the operator, --smooth-output, the CLI and the multi-GPU drivers in a one-rank group;
and the sideband selection of the whole chain."""
import os

import numpy as np
import pytest

import signals
from gpu_util import chunked
from oracle import oracle as orc
from sdrterm_b200.plan import build_plan
from ssb_ref import seamless_ssb_oracle, ssb, ssb_omega, ssb_oracle, ssb_sos
from util import parse_wav, rel_err

TOL = 1e-9
_ISZ = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'f': 4, 'd': 8}


def _kw(enc, q, iq, center, fs=1_024_000, norm=False, swap=False, simo=False, vfos=None, demod='usb', B=None):
    if B is None:
        B = min(5000, int(0.3 * (fs // q)))
    return dict(fs=fs, enc=enc, center=center, dec=q, demod=demod, omega_out=B, correct_iq=iq, vfos=vfos,
                simo=simo, normalize=norm, swap=swap, big_endian=None)


def _plan(kw, seamless=False):
    ch = orc.Chain(**{**kw, 'demod': 're'})
    return build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, simo=kw['simo'], swap=orc.needs_swap(ch.dt),
                      correct_iq=kw['correct_iq'], normalize=kw['normalize'], demod=kw['demod'],
                      omega_out=kw['omega_out'], seamless=seamless)


def _body(kw, nch, seed, extra=0):
    n = nch * 131072 // (2 * _ISZ[kw['enc']]) + extra
    return signals.generic_bytes(kw['enc'], n, seed, kw['fs'], kw['center'] or 40_000, big_endian=kw['swap'])


def _process(kw, body, use_tc=True, max_chunks=8):
    from sdrterm_b200.engine import Engine
    pl = _plan(kw)
    with Engine(pl, max_chunks=max_chunks, use_tc=use_tc) as eng:
        assert eng.W == pl.W == pl.M
        tc = eng.tc is not None
        out = np.asarray(eng.process(chunked(body)), dtype=np.float64)
    return out, pl, tc


# name, kw, use_tc, expected front end (True = k_tc)
CASES = [
    ('b d64 iq c20k', _kw('b', 64, True, 20000, fs=250_000), True, True),
    ('b-swap d64 lsb', _kw('b', 64, False, 20000, fs=250_000, swap=True, demod='lsb'), True, True),
    ('B d64 norm c0', _kw('B', 64, True, 0, fs=2_400_000, norm=True), True, False),
    ('B-swap d64 iq lsb', _kw('B', 64, True, -30000, fs=2_400_000, swap=True, demod='lsb'), True, True),
    ('h d64 iq k_tc', _kw('h', 64, True, 15000), True, True),
    ('h d64 iq k_tc lsb', _kw('h', 64, True, 15000, demod='lsb'), True, True),
    ('h d64 iq k_main', _kw('h', 64, True, 15000), False, False),
    ('h-swap d32 c0 lsb', _kw('h', 32, False, 0, swap=True, demod='lsb'), True, True),
    ('H d32 norm iq', _kw('H', 32, True, -50000, fs=1_000_000, norm=True), True, False),
    ('H-swap d32 iq lsb', _kw('H', 32, True, -50000, fs=1_000_000, swap=True, demod='lsb'), True, True),
    ('f d256 c30k', _kw('f', 256, False, 30000, fs=2_400_000), True, False),
    ('f-swap d64 iq lsb', _kw('f', 64, True, 30000, fs=2_400_000, swap=True, demod='lsb'), True, False),
    ('d d32 iq', _kw('d', 32, True, 12000, fs=192_000), True, False),
    ('d-swap d4 norm c0 lsb', _kw('d', 4, False, 0, fs=192_000, swap=True, norm=True, demod='lsb'), True, False),
    ('h d50 ragged iq', _kw('h', 50, True, 15000), True, False),
    ('h d50 ragged iq lsb', _kw('h', 50, True, 15000, demod='lsb'), True, False),
    ('B d25 odd iq', _kw('B', 25, True, 10000, fs=2_400_000), True, False),
    ('h d5 odd norm lsb', _kw('h', 5, False, 30000, norm=True, demod='lsb'), True, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,kw,use_tc,want_tc', CASES, ids=[c[0] for c in CASES])
def test_ssb_matches_oracle(name, kw, use_tc, want_tc):
    body = _body(kw, 2, 300 + kw['dec'], extra=1000)       # 3 chunks, the last one with a stale tail
    out, pl, tc = _process(kw, body, use_tc)
    assert tc == want_tc
    ref = ssb_oracle(kw, body)
    err = rel_err(out, ref)
    print(f'{name}: M={pl.M} B={kw["omega_out"]} err={err:.3e}')
    assert out.shape == ref.shape == (1, 3 * pl.M) and err < TOL


@pytest.mark.gpu
@pytest.mark.parametrize('demod', ['usb', 'lsb'])
@pytest.mark.parametrize('kw0', [_kw('h', 64, True, 15000), _kw('B', 64, True, 0, fs=2_400_000, norm=True)],
                         ids=['k_tc', 'k_main'])
def test_fused_and_general_paths_agree(kw0, demod, monkeypatch):
    kw = {**kw0, 'demod': demod}
    body = _body(kw, 3, 21)
    fused, pl, _ = _process(kw, body)
    monkeypatch.setenv('SDRB_NO_FINISH', '1')
    general, _, _ = _process(kw, body)
    err = rel_err(general, fused)
    print(f'{demod}: fused vs general {err:.3e}')
    assert err < 1e-11


@pytest.mark.gpu
def test_ssb_banks_match_oracle():
    """Config 3's 17-row big-endian SIMO bank (k_tc) and config 4's 257-row float32 bank (k_main)."""
    from sdrterm_b200.engine import Engine
    body, vfos = signals.c3_bytes(2 * 32768, seed=3)
    kw = _kw('h', 64, False, 0, fs=2_400_000, swap=True, simo=True, vfos=vfos)
    pl = _plan(kw)
    assert pl.R == 17 and pl.big_endian_out
    with Engine(pl, max_chunks=2) as eng:
        raw = eng.process(chunked(body))
        assert eng.tc is not None
    assert raw.dtype == np.dtype('>f8')
    ref = ssb_oracle(kw, body)
    err = rel_err(np.asarray(raw, dtype=np.float64), ref)
    print(f'17-row bank: err={err:.3e}')
    assert raw.shape == ref.shape and err < TOL
    body4, vfos4 = signals.c4_bytes(2 * 16384, seed=4)
    kw4 = _kw('f', 64, False, 0, fs=61_440_000, simo=True, vfos=vfos4, demod='lsb')
    pl4 = _plan(kw4)
    assert pl4.R == 257
    with Engine(pl4, max_chunks=2) as eng:
        out4 = np.asarray(eng.process(chunked(body4)), dtype=np.float64)
        assert eng.tc is None
    ref4 = ssb_oracle(kw4, body4)
    err4 = rel_err(out4, ref4)
    print(f'257-row bank: err={err4:.3e}')
    assert out4.shape == ref4.shape and err4 < TOL


@pytest.mark.gpu
def test_ssb_submit_wait_alternating_slots():
    from sdrterm_b200._native import PinnedBuffer
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, True, 15000)
    pl = _plan(kw)
    sizes = [1, 3, 2, 4, 1, 2, 3]
    body = _body(kw, sum(sizes), 5)
    cb = pl.chunk_bytes
    with Engine(pl, max_chunks=4) as eng:
        hin = [PinnedBuffer(4 * cb) for _ in range(2)]
        hout = [PinnedBuffer(eng.R * 4 * eng.W * 8) for _ in range(2)]
        parts, pending, o = [], [0, 0], 0

        def collect(s):
            eng.wait(s)
            parts.append(hout[s].view(np.float64)[:eng.W * pending[s]].copy())
            pending[s] = 0

        for b, n in enumerate(sizes):
            s = b & 1
            if pending[s]:
                collect(s)
            hin[s].u8[:n * cb] = np.frombuffer(body[o:o + n * cb], dtype=np.uint8)
            eng.submit(s, hin[s].ptr.value, n, hout[s].ptr.value)
            pending[s] = n
            o += n * cb
        collect(len(sizes) & 1)
        collect((len(sizes) - 1) & 1)
    out = np.concatenate(parts)[None]
    ref = ssb_oracle(kw, body)
    assert out.shape == ref.shape and rel_err(out, ref) < TOL


def _stream(eng, body, splits):
    cb = eng.chunk_bytes
    outs, o, i = [], 0, 0
    while o < len(body):
        k = splits[i % len(splits)]
        i += 1
        r = eng.stream(body[o:o + k * cb])
        assert r.shape[1] % eng.W == 0
        outs.append(np.asarray(r, dtype=np.float64))
        o += k * cb
    outs.append(np.asarray(eng.stream_end(), dtype=np.float64))
    return np.concatenate(outs, axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize('kw', [_kw('h', 64, True, 15000), _kw('f', 256, True, 30000, fs=2_400_000, demod='lsb')],
                         ids=['int16-d64-usb', 'float32-d256-lsb'])
def test_seamless_ssb_matches_oracle_across_batch_splits(kw):
    from sdrterm_b200.engine import Engine
    pl = _plan(kw, seamless=True)
    nch = 3 * (pl.lookahead + 1) + 2
    body = _body(kw, nch, 11)
    ref, _ = seamless_ssb_oracle(kw, body)
    res = []
    with Engine(pl, max_chunks=8) as eng:
        for split in (1, 2, 5, 8):
            out = _stream(eng, body, (split,))
            assert out.shape[1] == nch * pl.M
            res.append(out)
    worst = max(rel_err(o, res[0]) for o in res[1:])
    err = rel_err(res[0], ref)
    print(f'seamless {kw["demod"]} D={pl.lookahead}: err={err:.3e} split spread={worst:.3e}')
    assert worst <= 1e-12
    assert res[0].shape == ref.shape and err < TOL


@pytest.mark.gpu
def test_seamless_ssb_long_stream_and_bank():
    """A 300-chunk stream through many calls, and the 17-row big-endian bank, in seamless mode."""
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, True, 15000, demod='lsb')
    body = _body(kw, 300, 17)
    ref, _ = seamless_ssb_oracle(kw, body)
    with Engine(_plan(kw, seamless=True), max_chunks=16) as eng:
        out = _stream(eng, body, (16, 7, 13))
    err = rel_err(out, ref)
    print(f'seamless 300 chunks: err={err:.3e}')
    assert out.shape == ref.shape and err < TOL
    body3, vfos = signals.c3_bytes(4 * 32768, seed=3)
    kw3 = _kw('h', 64, False, 0, fs=2_400_000, swap=True, simo=True, vfos=vfos)
    with Engine(_plan(kw3, seamless=True), max_chunks=4) as eng:
        out3 = _stream(eng, body3, (3, 1))
    ref3, _ = seamless_ssb_oracle(kw3, body3)
    assert out3.shape == ref3.shape and rel_err(out3, ref3) < TOL


def _tones(fs, center, lines, n, enc='f'):
    """Complex tones (offset from `center` in Hz, amplitude) as raw interleaved samples."""
    k = np.arange(n)
    z = sum(a * np.exp(2j * np.pi * ((center + f) / fs) * k) for f, a in lines)
    iq = np.empty(2 * n, dtype=np.float32 if enc == 'f' else np.int16)
    scale = 1.0 if enc == 'f' else 8000.0
    iq[0::2], iq[1::2] = np.real(z) * scale, np.imag(z) * scale
    return iq.tobytes()


@pytest.mark.gpu
def test_seamless_tone_is_smooth_across_chunk_edges():
    """A steady in-band tone: the seamless output fits one sinusoid at every chunk edge; the default
    mode restarts the filter at each chunk and shows its transient there."""
    from sdrterm_b200.engine import Engine
    fs, q, fc = 1_024_000, 64, 15000
    nch = 8
    kw = _kw('f', q, False, fc, fs=fs, B=3000)
    body = _tones(fs, fc, [(1000, 0.5)], nch * 32768)
    outs = {}
    for sm in (False, True):
        pl = _plan(kw, seamless=sm)
        with Engine(pl, max_chunks=nch) as eng:
            outs[sm] = _stream(eng, body, (3,))[0] if sm else np.asarray(eng.process(body), dtype=np.float64)[0]
    M = pl.M
    k = np.arange(outs[True].size)
    w = 2 * np.pi * 1000 / (fs // q)
    sel = (k >= 2 * M) & (k < (nch - 1) * M)
    X = np.stack([np.cos(w * k), np.sin(w * k)], axis=1)
    coef = np.linalg.lstsq(X[sel], outs[True][sel], rcond=None)[0]
    fit = X @ coef
    amp = np.hypot(*coef)
    edges = np.concatenate([np.arange(c * M - 2, c * M + 3) for c in range(2, nch - 1)])
    dev_seam = np.max(np.abs(outs[True][edges] - fit[edges])) / amp
    dev_std = np.max(np.abs(outs[False][edges] - fit[edges])) / amp
    print(f'edge deviation: seamless {dev_seam:.2e}, default {dev_std:.2e} (of the tone amplitude)')
    assert dev_seam < 1e-4 and dev_std > 0.1


@pytest.mark.gpu
def test_chain_selects_the_sideband():
    """Tones at VFO + 1 kHz and VFO - 1.5 kHz through the whole chain: usb audio holds the 1 kHz line
    with the 1.5 kHz one >= 25 dB down, lsb the reverse."""
    from sdrterm_b200.engine import Engine
    fs, q, fc = 1_024_000, 64, 15000
    fs_d = fs // q
    body = _tones(fs, fc, [(1000, 0.3), (-1500, 0.3)], 6 * 32768, enc='h')
    lvl = {}
    for demod in ('usb', 'lsb'):
        kw = _kw('h', q, False, fc, fs=fs, demod=demod, B=3000)
        pl = _plan(kw)
        with Engine(pl, max_chunks=6) as eng:
            s = np.asarray(eng.process(body), dtype=np.float64)[0].reshape(-1, pl.M)
        # the line amplitudes by least squares over the settled second half of every chunk (each
        # chunk restarts the NCO and the filter)
        k = np.arange(pl.M // 2, pl.M)
        X = np.stack([g(2 * np.pi * f / fs_d * k) for f in (1000, 1500) for g in (np.cos, np.sin)], axis=1)
        amp = np.zeros(2)
        for row in s:
            c = np.linalg.lstsq(X, row[pl.M // 2:], rcond=None)[0]
            amp += np.hypot(c[0::2], c[1::2]) / len(s)
        lvl[demod] = {1000: 20 * np.log10(amp[0]), 1500: 20 * np.log10(amp[1])}
    print(lvl)
    assert lvl['usb'][1000] - lvl['usb'][1500] >= 25
    assert lvl['lsb'][1500] - lvl['lsb'][1000] >= 25


@pytest.mark.gpu
@pytest.mark.parametrize('M', [512, 1311])
@pytest.mark.parametrize('demod', ['usb', 'lsb'])
def test_ssb_operator_matches_oracle(M, demod):
    from sdrterm_b200.dsp import demodulation as dem
    rng = np.random.default_rng(M)
    y = rng.normal(size=(3, M)) + 1j * rng.normal(size=(3, M))
    sos, om = ssb_sos(1_024_000, 64, 3000), ssb_omega(demod, 3000, 16000)
    res = np.empty((3, M))
    (dem.usbDemod if demod == 'usb' else dem.lsbDemod)(y, res, sos, om)
    ref = ssb(y, sos, om)
    err = rel_err(res, ref)
    print(f'operator {demod} M={M}: err={err:.3e}')
    assert err < TOL
    one = ssb_sos(1_024_000, 64, 3000)[:1]
    dem.ssbDemod(y, res, one, om)                          # a one-section prototype
    assert rel_err(res, ssb(y, one, om)) < TOL


@pytest.mark.gpu
def test_ssb_smoothing_matches_savgol_of_the_oracle():
    from scipy.signal import savgol_filter
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, True, 15000)
    body = _body(kw, 3, 8)
    pl = _plan(kw)
    with Engine(pl, max_chunks=4, smooth=9) as eng:
        out = np.asarray(eng.process(chunked(body)), dtype=np.float64)
    ref = ssb_oracle(kw, body).reshape(-1, pl.M)
    ref = np.stack([savgol_filter(r, 9, 3) for r in ref]).reshape(1, -1)
    err = rel_err(out, ref)
    print(f'smoothed usb: err={err:.3e}')
    assert err < TOL


def _cli_env():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return dict(os.environ, PYTHONPATH=os.path.join(root, 'src'))


@pytest.mark.gpu
def test_cli_usb_wav_matches_oracle(tmp_path):
    import subprocess
    import sys
    raw = signals.c1_bytes(3 * 32768 + 5000, seed=0)
    fin, fout = tmp_path / 'in.wav', tmp_path / 'out.bin'
    fin.write_bytes(raw)
    subprocess.run([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-o', str(fout), '-c', '15000',
                    '-d', '64', '-m', 'usb', '-w', '3000', '--correct-iq'], env=_cli_env(), cwd=str(tmp_path),
                   check=True, timeout=300, capture_output=True)
    fs, enc, be, off = parse_wav(raw)
    kw = _kw(enc, 64, True, 15000, fs=fs, B=3000)
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')[None]
    ref = ssb_oracle(kw, raw[off:])
    assert got.shape == ref.shape == (1, 4 * 512)
    assert rel_err(got, ref) < TOL


@pytest.mark.gpu
def test_cli_simo_lsb_sockets(tmp_path):
    """`--simo -m lsb`: every VFO socket receives M big-endian doubles per chunk, its row of the oracle."""
    import socket
    import subprocess
    import sys
    import threading
    import time
    nch = 3
    body, vfos = signals.c3_bytes(nch * 32768, seed=3)
    vf = ','.join(vfos.split(',')[:2])
    fin = tmp_path / 'in.raw'
    fin.write_bytes(body)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    proc = subprocess.Popen([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-r', '2400k', '-e', 'h', '-X', '-d', '64',
                             '-m', 'lsb', '-w', '5000', '--simo', f'--vfos={vf}', '--vfo-host', f'127.0.0.1:{port}'],
                            env=_cli_env(), cwd=str(tmp_path), stderr=subprocess.PIPE, text=True)
    head = ''
    deadline = time.time() + 120
    while time.time() < deadline and 'Accepting' not in head:
        line = proc.stderr.readline()
        if not line:
            break
        head += line
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
    kw = _kw('h', 64, False, 0, fs=2_400_000, swap=True, simo=True, vfos=vf, demod='lsb', B=5000)
    ref = ssb_oracle(kw, body)
    M = 32768 // 64
    assert sorted(got) == [0, 1, 2]
    for i in range(3):
        assert len(got[i]) == nch * M * 8
        g = np.frombuffer(got[i], dtype='>f8').astype(np.float64)
        assert min(rel_err(g, r) for r in ref) < TOL


@pytest.mark.gpu
def test_multigpu_drivers_carry_ssb_rows_in_a_one_rank_group(tmp_path):
    import torch
    import torch.distributed as dist
    from sdrterm_b200 import multigpu
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, True, 15000, B=3000)
    pl = _plan(kw)
    nch = 3
    body = signals.c1_bytes(nch * 32768, seed=9, header=False)
    with Engine(pl, max_chunks=nch) as eng:
        want = np.asarray(eng.process(body), dtype=np.float64)
    assert rel_err(want, ssb_oracle(kw, body)) < TOL
    dist.init_process_group('gloo', init_method=f'file://{tmp_path}/pg', rank=0, world_size=1)
    try:
        dev = torch.device('cuda', 0)
        raw = torch.from_numpy(np.frombuffer(body, dtype=np.uint8).copy()).to(dev)
        chain = multigpu.TimeShardedChain(pl, max_chunks=nch, device=0, dist=dist, torch=torch)
        out = torch.empty((1, nch * pl.W), dtype=torch.float64, device=dev)
        chain.step(raw.data_ptr(), nch, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        chain.close()
        assert np.array_equal(out.cpu().numpy(), want)
        path = tmp_path / 'in.raw'
        path.write_bytes(body)
        got = multigpu.run_file_sharded(str(path), None, fs=1_024_000, enc='h', dec=64, center=15000, demod='usb',
                                        omega_out=3000, correct_iq=True, batch_chunks=2, device=0, dist=dist,
                                        torch=torch)
        assert got.shape == want.shape and rel_err(got, want) < 1e-13
        bvfos = [100_000, -200_000]
        bank = multigpu.RowShardedBank(2_400_000, 'h', 64, bvfos + [0], max_chunks=nch, device=0, dist=dist, torch=torch,
                                       demod='lsb', omega_out=5000)
        assert bank.W == bank.M
        outs = [torch.empty((3, nch * bank.W), dtype=torch.float64, device=dev)]
        bank.run([raw], nch, outs, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        bank.close()
        bkw = _kw('h', 64, False, 0, fs=2_400_000, simo=True, vfos=','.join(str(v) for v in bvfos), demod='lsb', B=5000)
        bref = ssb_oracle(bkw, body)
        bgot = outs[0].cpu().numpy().view('>f8').astype(np.float64)
        assert bgot.shape == bref.shape and rel_err(bgot, bref) < TOL
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize('seamless', [False, True], ids=['default', 'seamless'])
def test_ssb_step_launches_as_many_kernels_as_fm(seamless, monkeypatch):
    from sdrterm_b200.engine import Engine
    counts = {}
    for general in (False, True):
        if general:
            monkeypatch.setenv('SDRB_NO_FINISH', '1')
        for demod in ('fm', 'usb', 'lsb'):
            kw = _kw('h', 64, True, 15000, demod=demod, B=3000)
            body = _body(kw, 4, 2)
            with Engine(_plan(kw, seamless=seamless), max_chunks=4) as eng:
                n0 = eng.launches
                if seamless:
                    eng.stream(body)
                    eng.stream_end()
                else:
                    eng.process(body)
                counts[general, demod] = eng.launches - n0
    print(counts)
    for general in (False, True):
        assert counts[general, 'usb'] == counts[general, 'lsb'] == counts[general, 'fm']
