"""GPU: the reference-facing host layer end to end -- CLI, processors, module operators --
against the oracle, the reference's golden outputs and the reference's own known-answer vectors
(test/dsp/demodulation_test.py:14-50)."""
import math
import queue
import socket
import threading

import numpy as np
import pytest
from scipy.signal import resample

from cases import CASES
from oracle import oracle as orc
from util import case_stream, load_golden, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-9


class Flag:
    value = 0


def test_cli_readme_example_matches_reference_golden(tmp_path):
    """BASELINE config 1: int16 IQ WAV at 1024 kS/s, -c 15k -w 5k -d 64 --correct-iq, float64 out."""
    from sdrterm_b200.sdrterm import main
    raw, body, kw = case_stream('c1_fm_wav_int16')
    fin, fout = tmp_path / 'in.wav', tmp_path / 'out.bin'
    fin.write_bytes(raw)
    assert main(['-i', str(fin), '-o', str(fout), '-c', '15k', '-w', '5k', '-d', '64', '--correct-iq']) == 0
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')
    g = load_golden('c1_fm_wav_int16')
    assert got.shape == g['out'][0].shape              # incl. the stale-tail chunk (8-Q5)
    assert rel_err(got, g['out'][0]) < TOL


def test_cli_raw_u8_am_d50(tmp_path):
    """BASELINE config 2 (-d 50: ceil(N/q) outputs per chunk, SURVEY 8-Q1)."""
    from sdrterm_b200.sdrterm import main
    raw, body, kw = case_stream('c2_am_u8_d50_ceil')
    fin, fout = tmp_path / 'in.raw', tmp_path / 'out.bin'
    fin.write_bytes(raw)
    assert main(['-i', str(fin), '-o', str(fout), '-r', '2400k', '-e', 'B', '-d', '50', '-w', '5k', '-m', 'am',
                 '--correct-iq']) == 0
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')
    g = load_golden('c2_am_u8_d50_ceil')
    assert got.shape == g['out'][0].shape and rel_err(got, g['out'][0]) < TOL


def test_processor_accepts_the_reference_queue_payload(tmp_path):
    """Chunks as the reference's producer sends them: decoded, IQ-corrected complex128 arrays."""
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    raw, body, kw = case_stream('c1_fm_wav_int16')
    ch = orc.Chain(**kw)
    n = len(body) // 131072
    zs = [ch.ingest(body[c * 131072:(c + 1) * 131072]).copy() for c in range(n)]
    ch2 = orc.Chain(**kw)
    yy = ch2.decimated(np.stack(zs))
    ref = np.concatenate([ch2.demodulate(yy[c]) for c in range(n)], axis=1)
    p = DspProcessor(kw['fs'], center=kw['center'], omegaOut=kw['omega_out'], dec=kw['dec'])
    p.selectOutputFm()
    q = queue.Queue()
    for z in zs:
        q.put(z)
    q.put(b'')
    fout = tmp_path / 'o.bin'
    p.processData(Flag(), q, str(fout))
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')
    assert got.shape == ref[0].shape and rel_err(got, ref[0]) < TOL


def test_simo_rows_over_sockets_big_endian():
    from sdrterm_b200.dsp.vfo_processor import VfoProcessor
    import signals
    body, vfos = signals.c3_bytes(2 * 32768, seed=3)
    vf = [int(v) for v in vfos.split(',')[:2]]
    kw = dict(fs=2_400_000, enc='h', center=0, dec=64, demod='fm', omega_out=5000, correct_iq=False,
              vfos=','.join(map(str, vf)), simo=True, normalize=False, swap=True, big_endian=None)
    ref = orc.Chain(**kw).run(body)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    p = VfoProcessor(2_400_000, vfoHost=f'127.0.0.1:{port}', vfos=','.join(map(str, vf)), dec=64, omegaOut=5000,
                     enc='h', swapEndianness=True)
    p.selectOutputFm()
    q = queue.Queue()
    for c in range(len(body) // 131072):
        q.put(body[c * 131072:(c + 1) * 131072])
    q.put(b'')
    th = threading.Thread(target=p.processData, args=(Flag(), q), daemon=True)
    th.start()
    got = {}

    def client(i):
        for _ in range(100):
            try:
                c = socket.create_connection(('127.0.0.1', port), timeout=5)
                break
            except OSError:
                import time
                time.sleep(0.1)
        need = ref.shape[1] * 8
        buf = b''
        while len(buf) < need:
            d = c.recv(need - len(buf))
            if not d:
                break
            buf += d
        got[i] = np.frombuffer(buf, dtype='>f8')
        c.close()

    cl = [threading.Thread(target=client, args=(i,), daemon=True) for i in range(3)]
    for t in cl:
        t.start()
    for t in cl:
        t.join(60)
    th.join(60)
    assert len(got) == 3
    # clients are handed rows in connection order, which threads do not fix: match as a set
    rows = [np.asarray(ref[r], dtype=np.float64) for r in range(3)]
    for i in range(3):
        assert got[i].shape == rows[0].shape
        assert min(rel_err(got[i], r) for r in rows) < TOL


def test_module_operators_known_answers():
    """The reference's own 8-sample vector: fm/am within 1e-12, re/im exact."""
    import sdrterm_b200.dsp.demodulation as dem
    inp = np.array([[0j, 1 + 2j, 2 + 3j, 3 + 4j, 4 + 5j, 5 + 6j, 6 + 7j, 7 + 8j]])
    out = np.empty((1, 8))
    dem.fmDemod(inp, out)
    exp = [0.0] * 4
    for i in range(0, 8, 2):
        t = inp[0][i] * inp[0][i + 1].conjugate()
        exp[i >> 1] = math.atan2(t.imag, t.real)
    exp = resample(exp, 8)
    assert np.max(np.abs(out[0] - exp)) < 1e-12
    dem.amDemod(inp, out)
    assert np.max(np.abs(out[0] - np.array([z.real ** 2 + z.imag ** 2 for z in inp[0]]))) < 1e-12
    dem.realOutput(inp, out)
    assert np.array_equal(out[0], inp[0].real)
    dem.imagOutput(inp, out)
    assert np.array_equal(out[0], inp[0].imag)
    rng = np.random.default_rng(0)
    y = rng.normal(size=64) + 1j * rng.normal(size=64)
    sh = np.exp(-2j * np.pi * rng.random((3, 64)))
    res = np.empty((3, 64), dtype=np.complex128)
    dem.shiftFreq(y, sh, res)
    assert np.max(np.abs(res - y * sh)) < 1e-15
    with pytest.raises(ValueError):
        dem.amDemod(inp, np.empty((2, 8)))


def test_fm_demod_operator_takes_any_even_length():
    """demodulation.py:35-38 resamples for any n; rows of 2*2^k (k >= 1) take the FFT path,
    everything else the dense resample matrix (ADVICE r1).  2: the matrix; 4: no FFT pass; 8: one
    radix-2 pass; 16: one radix-4 pass; 2048 / 4096: shared / global scratch; 16384."""
    import sdrterm_b200.dsp.demodulation as dem
    rng = np.random.default_rng(3)
    for n in (2, 4, 6, 8, 10, 16, 24, 100, 1310, 512, 2048, 4096, 16384):
        y = rng.normal(size=(2, n)) + 1j * rng.normal(size=(2, n))
        out = np.empty((2, n))
        dem.fmDemod(y, out)
        ref = np.stack([resample(np.angle(r[0::2] * np.conj(r[1::2])), n) for r in y])
        assert np.max(np.abs(out - ref)) < 1e-11, n
    with pytest.raises(Exception):
        dem.fmDemod(rng.normal(size=(1, 7)) + 0j, np.empty((1, 7)))


def test_iq_correction_plugin_matches_the_serial_recurrence():
    """dsp.fast.iq_correction.IQCorrection.correctIq vs the loop of read_file.py:72-77, state
    carried across calls (the reference's own test allows 10E-2; here 1e-12 relative)."""
    from sdrterm_b200.dsp.fast.iq_correction import IQCorrection
    rng = np.random.default_rng(8)
    fs = 1_024_000
    c = IQCorrection(fs)
    off = np.zeros(1, dtype=np.complex128)
    roff = 0j
    L = 50 / fs
    for n in (32768, 1000, 65536):
        z = (rng.normal(size=n) * 8000 + 37) + 1j * (rng.normal(size=n) * 8000 - 21)
        ref = z.copy()
        for i in range(n):
            ref[i] -= roff
            roff += ref[i] * L
        c.correctIq(z, off)
        assert np.max(np.abs(z - ref)) <= 1e-12 * np.max(np.abs(ref))
        assert abs(off[0] - roff) <= 1e-12 * max(1.0, abs(roff))


def test_cli_simo_prints_the_lines_example_simo_scrapes(tmp_path):
    """example_simo.sh reads stderr for the repr JSON keys (host, vfos, tunedFreq, decimatedFs),
    then `Accepting connections on ('<ip>', <port>)`, attaches one client per row and waits for
    `Connection(s) established` (example_simo.sh:96-118,165-170; src/sdrterm.py:144,
    vfo_processor.py:78,110).  Run the drop-in CLI as a subprocess the same way."""
    import json
    import os
    import re
    import subprocess
    import sys
    import time
    import signals
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    body, vfos = signals.c3_bytes(2 * 32768, seed=3)
    vf = vfos.split(',')[:2]
    fin = tmp_path / 'in.raw'
    fin.write_bytes(body)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    env = dict(os.environ, PYTHONPATH=os.path.join(root, 'src'))
    proc = subprocess.Popen([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-r', '2400k', '-e', 'h', '-X', '-d', '64',
                             '-w', '5k', '--simo', f'--vfos={",".join(vf)}', '--vfo-host', f'127.0.0.1:{port}',
                             '-t', '155685000'],
                            env=env, cwd=str(tmp_path), stderr=subprocess.PIPE, text=True)
    lines = []
    deadline = time.time() + 120
    while time.time() < deadline:
        line = proc.stderr.readline()
        if not line:
            break
        lines.append(line)
        if 'Accepting' in line:
            break
    head = ''.join(lines)
    m = re.search(r"Accepting connections on \('127\.0\.0\.1', (\d+)\)", head)
    assert m and int(m.group(1)) == port, head
    d = json.loads(head[head.index('{'):head.rindex('}') + 1])
    assert d['vfos'] == ','.join(vf) + ',0' and d['host'] == '127.0.0.1' and d['tunedFreq'] == 155685000
    assert d['decimatedFs'] == 2_400_000 // 64
    got = {}

    def client(i):
        c = socket.create_connection(('127.0.0.1', port), timeout=30)
        buf = b''
        while True:
            dta = c.recv(1 << 16)
            if not dta:
                break
            buf += dta
        got[i] = np.frombuffer(buf[:len(buf) // 8 * 8], dtype='>f8')
        c.close()

    cl = [threading.Thread(target=client, args=(i,), daemon=True) for i in range(3)]
    for t in cl:
        t.start()
    rest = proc.stderr.read()
    proc.wait(120)
    for t in cl:
        t.join(30)
    assert 'Connection(s) established' in rest, rest
    assert proc.returncode == 0
    kw = dict(fs=2_400_000, enc='h', center=0, dec=64, demod='fm', omega_out=5000, correct_iq=False,
              vfos=','.join(vf), simo=True, normalize=False, swap=True, big_endian=None)
    ref = orc.Chain(**kw).run(body)
    rows = [np.asarray(ref[r], dtype=np.float64) for r in range(3)]
    assert len(got) == 3
    for i in range(3):
        assert got[i].shape == rows[0].shape
        assert min(rel_err(got[i], r) for r in rows) < TOL


@pytest.mark.parametrize('window', [5, 11, 32])
def test_cli_smooth_output_matches_savgol_per_chunk(tmp_path, window):
    """--smooth-output N: dsp_processor.py:159-160 applies savgol_filter(z, N, 3) to every chunk's
    output row after the output low-pass (standard mode only)."""
    from scipy.signal import savgol_filter
    from sdrterm_b200.sdrterm import main
    raw, body, kw = case_stream('c1_fm_wav_int16')
    fin, fout = tmp_path / 'in.wav', tmp_path / 'out.bin'
    fin.write_bytes(raw)
    assert main(['-i', str(fin), '-o', str(fout), '-c', '15k', '-w', '5k', '-d', '64', '--correct-iq',
                 '--smooth-output', str(window)]) == 0
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')
    g = load_golden('c1_fm_wav_int16')['out'][0]
    M = 512
    ref = np.concatenate([savgol_filter(g[c * M:(c + 1) * M], window, 3) for c in range(g.size // M)])
    assert got.shape == ref.shape and rel_err(got, ref) < TOL


def _db_close(got, want, floor_db, tol):
    """Decibel-type outputs: compare where the reference is above `floor_db` below its maximum (a
    bin that is numerically zero has an ill-conditioned logarithm), and the linear values everywhere."""
    assert got.shape == want.shape
    top = want.max()
    big = want > top - floor_db
    assert np.abs(got[big] - want[big]).max() <= tol
    return np.abs(got[big] - want[big]).max()


@pytest.mark.parametrize('n', [8192, 16384, 32768, 65536])
def test_power_spectrum_feed_matches_the_plot_arithmetic(n):
    """SURVEY 8-f3: SpectrumAnalyzerPlot.update (spectrum_analyzer_plot.py:75-92) on the device:
    log10(|fftshift(fftn(y*shift, norm='forward'))|^2) and the frequency axis."""
    from scipy.fft import fftfreq, fftshift
    from sdrterm_b200.plots import SpectrumFeed, powerSpectrum
    rng = np.random.default_rng(n)
    fs, center = 1_024_000, 15_000
    t = np.arange(n)
    y = 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) + np.exp(2j * np.pi * 0.11 * t) + 0.3
    feed = SpectrumFeed(fs, center=center)
    freq, amp = feed.update(y)
    want = orc.power_spectrum(y, orc.plot_shift(center, fs, n))
    assert np.array_equal(freq, fftshift(fftfreq(n, 1 / fs)))
    # linear power, relative to the strongest bin: 1e-12; decibels down to 100 dB below it: 1e-9
    assert np.abs(10 ** amp - 10 ** want).max() <= 1e-12 * (10 ** want).max()
    _db_close(amp, want, 10.0, 1e-9)
    # batch of rows, no shift
    rows = np.stack([y, y[::-1], 2 * y])
    got = powerSpectrum(rows)
    for r in range(3):
        _db_close(got[r], orc.power_spectrum(rows[r], None), 10.0, 1e-9)


def test_power_spectrum_feed_rejects_what_it_cannot_do():
    from sdrterm_b200._native import SdrbError
    from sdrterm_b200.plots import powerSpectrum
    with pytest.raises(SdrbError):
        powerSpectrum(np.ones(1000, dtype=np.complex128))          # not a power of two
    with pytest.raises(ValueError):
        powerSpectrum(np.ones(1024, dtype=np.complex128), shift=np.ones(8))


@pytest.mark.parametrize('n', [1000, 16384, 32768])
def test_waterfall_feed_matches_short_time_fft(n):
    """SURVEY 8-f3: WaterfallPlot.update (waterfall_plot.py:90-99) on the device against SciPy's
    ShortTimeFFT itself (the reference's call) and the oracle's restatement."""
    from scipy.signal import ShortTimeFFT
    from sdrterm_b200.plots import WaterfallFeed
    rng = np.random.default_rng(n)
    fs, center = 1_024_000, -20_000
    t = np.arange(n)
    y = 0.1 * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) + np.exp(2j * np.pi * (0.05 + 1e-6 * t) * t)
    feed = WaterfallFeed(fs, center=center)
    img = feed.update(y)
    S = ShortTimeFFT.from_window(('kaiser', 5), fs, 256, 128, mfft=1024, fft_mode='centered', scale_to='magnitude',
                                 phase_shift=None)
    sh = orc.plot_shift(center, fs, n)
    want = 10. * np.log10(abs(S.stft(y * sh)))
    assert img.shape == want.shape == (1024, n // 128 + 1 if n % 128 == 0 else S.p_max(n))
    _db_close(img, want, 60.0, 1e-8)
    _db_close(img, orc.stft_db(y, sh, S.win, S.hop, 1024, S.p_max(n)), 60.0, 1e-8)


@pytest.mark.parametrize('enc,flags,kwx', [
    ('h', ['-d', '25', '-m', 'am', '--correct-iq'], dict(dec=25, demod='am', correct_iq=True)),
    ('f', ['-d', '64', '-m', 'fm', '--center-frequency=-20k'], dict(dec=64, demod='fm', center=-20000)),
    ('H', ['-d', '32', '-m', 're', '-X', '--correct-iq', '-c', '12k'], dict(dec=32, demod='re', swap=True, correct_iq=True, center=12000)),
    ('b', ['-d', '128', '-m', 'im', '--normalize-input'], dict(dec=128, demod='im', normalize=True)),
    ('i', ['-d', '128', '-m', 'fm', '--correct-iq'], dict(dec=128, demod='fm', correct_iq=True)),
    ('d', ['-d', '16', '-m', 'am', '-c', '30k'], dict(dec=16, demod='am', center=30000)),
])
def test_cli_option_sweep_on_raw_files(tmp_path, enc, flags, kwx):
    """Raw files through the CLI (reader thread -> page-locked chunk pool -> double-buffered
    processor -> file writer) for options the named configs do not combine; 9 chunks plus a short
    one, so the batches are 9 whole chunks read at once and the stale tail of the last (8-Q5)."""
    import signals
    from sdrterm_b200.sdrterm import main
    isz = {'b': 1, 'h': 2, 'H': 2, 'i': 4, 'f': 4, 'd': 8}[enc]
    n = 9 * (131072 // (2 * isz)) + 1000
    swap = bool(kwx.get('swap'))
    body = signals.generic_bytes(enc, n, 77, 1_000_000, kwx.get('center', 0) or 40_000, big_endian=swap)
    fin, fout = tmp_path / 'in.raw', tmp_path / 'out.bin'
    fin.write_bytes(body)
    assert main(['-i', str(fin), '-o', str(fout), '-r', '1M', '-e', enc, '-w', '3k'] + flags) == 0
    kw = dict(fs=1_000_000, enc=enc, center=0, dec=2, demod='fm', omega_out=3000, correct_iq=False, vfos=None, simo=False,
              normalize=False, swap=False, big_endian=None)
    kw.update(kwx)
    ref = orc.Chain(**kw).run(body)
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')
    assert got.shape == ref[0].shape and rel_err(got, ref[0]) < TOL
