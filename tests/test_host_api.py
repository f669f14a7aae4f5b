"""Host-side mirror of the reference's processor / ingest API (no GPU needed): the cases of the
reference's own test/dsp/dsp_processor_test.py:21-75, test/misc/read_file_test.py and
test/misc/file_util_test.py that concern this path, against sdrterm_b200.dsp / .misc and the
``src/`` import shims."""
import io
import math
import os
import pickle
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

import sdrterm_b200.dsp.demodulation as dem
import sdrterm_b200.dsp.dsp_processor as dsp
from sdrterm_b200.dsp.data_processor import DataProcessor
from sdrterm_b200.dsp.vfo_processor import VfoProcessor
from sdrterm_b200.misc import file_util, read_file

FS, CENTER, NSHIFT, DEC = 48000, -1000, 8, 3


def test_processor_surface_like_reference():
    p = dsp.DspProcessor(FS, omegaOut=250)
    assert p.fs == FS and p.decimation == 2 and p.decimatedFs == FS >> 1
    p.selectOutputFm()
    assert p.demod == dem.fmDemod and p.bandwidth == 12500 and len(p._outputFilters) == 2
    p.selectOutputAm()
    assert p.demod == dem.amDemod and p.bandwidth == 10000
    p.selectOutputReal()
    assert p.demod == dem.realOutput and p._outputFilters == [] and p.bandwidth == p.decimatedFs
    p.selectOutputImag()
    assert p.demod == dem.imagOutput
    with pytest.raises(ValueError):
        p.decimation = 1
    with pytest.raises(AttributeError):
        p.decimatedFs = 1
    with pytest.raises(ValueError):
        p._setDemod(None, ())
    with pytest.raises(TypeError):
        p._setDemod('asdf', None)
    p.decimation = DEC
    assert p.decimation == DEC and p.decimatedFs == FS / DEC
    p._generateShift(NSHIFT)
    assert p._shift is None                       # centre 0: no shift (dsp_processor.py:185-187)
    p.centerFreq = CENTER
    p._generateShift(NSHIFT)
    assert p._shift.size == NSHIFT
    for k in range(NSHIFT):
        assert p._shift[0][k] == np.pow(math.e, -2j * math.pi * (CENTER / FS) * k)
    with pytest.raises(FileNotFoundError):
        p.processData(None, None, '')
    with pytest.raises(AttributeError):
        p.processData(None, None, None)
    with pytest.raises(TypeError):
        DataProcessor()
    DataProcessor.processData(None)


def test_processor_pickles_without_cuda_state():
    p = dsp.DspProcessor(1_024_000, center=15000, omegaOut=5000, dec=64, enc='h', correctIq=True)
    p.selectOutputFm()
    q = pickle.loads(pickle.dumps(p))
    assert q.fs == p.fs and q.decimation == 64 and q.demod == dem.fmDemod and q._engine is None
    assert 'decimatedFs' in repr(q)


def test_vfo_processor_rows_and_errors():
    with pytest.raises(ValueError):
        VfoProcessor(2_400_000, vfos=None)
    with pytest.raises(ValueError):
        VfoProcessor(2_400_000, vfos='')
    v = VfoProcessor(2_400_000, vfoHost='127.0.0.1:0', vfos='-100000,200000', center=5000, dec=64)
    assert list(v.vfos) == [-95000, 205000, 5000] and v._nFreq == 3     # centre appended (8-Q9)
    assert v.host == '127.0.0.1' and v.port == 0 and v.vfosStr == '-100000,200000,0'
    v._generateShift(4)
    w = -2j * np.pi * (v.vfos / v.fs)
    assert np.array_equal(v._shift, np.exp(w[:, None] * np.arange(4)[None, :]))
    v2 = VfoProcessor(2_400_000, vfoHost='127.0.0.1', vfos='1')
    assert v2.port > 0


def test_generate_domain_table():
    """test/misc/read_file_test.py:12-19."""
    assert read_file.generateDomain('B') == (0, 1 / 255)
    assert read_file.generateDomain('b') == (-128, 1 / 255)
    assert read_file.generateDomain('h') == (-32768, 1 / 65535)
    assert read_file.generateDomain('H') == (0, 1 / 65536)
    assert read_file.generateDomain('i') == (-2147483648, 1 / 4294967295)
    assert read_file.generateDomain('I') == (0, 1 / 4294967295)
    assert read_file.generateDomain('f') is None and read_file.generateDomain('d') is None


def _wav(tmp_path, tag=b'RIFF', fmt=1, bits=16, rate=1_024_000, payload=b'\x01\x02' * 64):
    e = '<' if tag == b'RIFF' else '>'
    hdr = tag + struct.pack(e + 'I', 36 + len(payload)) + b'WAVEfmt ' + \
        struct.pack(e + 'IHHIIHH', 16, fmt, 2, rate, rate * 2 * bits // 8, 2 * bits // 8, bits) + \
        b'data' + struct.pack(e + 'I', len(payload)) + payload
    f = tmp_path / 'x.wav'
    f.write_bytes(hdr)
    return str(f)


def test_wav_header_and_offset_quirk(tmp_path):
    info = file_util.checkWavHeader(_wav(tmp_path), None, None)
    assert info['sampRate'] == 1_024_000 and info['bitsPerSample'] == np.dtype('<i2')
    assert info['dataOffset'] == 40 and not info['isSocket']        # 4 bytes short of 44 (8-Q4)
    info = file_util.checkWavHeader(_wav(tmp_path, tag=b'RIFX'), None, None)
    assert info['bitsPerSample'] == np.dtype('>i2')
    info = file_util.checkWavHeader(_wav(tmp_path, fmt=3, bits=32), None, None)
    assert info['bitsPerSample'] == np.dtype('<f4')
    info = file_util.checkWavHeader(_wav(tmp_path, bits=8), None, None)
    assert info['bitsPerSample'] == np.dtype('u1')
    with pytest.raises(ValueError):
        file_util.checkWavHeader(_wav(tmp_path, fmt=7), None, None)


def test_raw_type_rules(tmp_path):
    raw = tmp_path / 'x.raw'
    raw.write_bytes(b'\0' * 64)
    info = file_util.checkWavHeader(str(raw), 2_400_000, 'B')
    assert info['bitsPerSample'] == np.dtype('u1') and info['dataOffset'] == 0
    with pytest.raises(ValueError):
        file_util.checkWavHeader(str(raw), None, 'B')
    with pytest.raises(ValueError):
        file_util.parseRawType(None, 1000, None)
    assert file_util.parseRawType('host:1234', 1000, 'h', True)['bitsPerSample'] == np.dtype('>i2')
    assert file_util.parseIntString('15k') == 15000 and file_util.parseIntString('2.4M') == 2_400_000
    assert file_util.parseIntString('64') == 64 and file_util.parseIntString(7) == 7


def test_chunk_reader_reuses_its_buffer_like_the_reference():
    """A short final read leaves the previous chunk's tail in the buffer and the whole buffer is
    processed (SURVEY 8-Q5)."""
    data = bytes(range(256)) * 4 + b'\xff' * 100
    got = list(read_file.chunks(io.BytesIO(data), readSize=512))
    assert len(got) == 3
    assert got[0].tobytes() == data[:512] and got[1].tobytes() == data[512:1024]
    assert got[2].tobytes() == b'\xff' * 100 + data[512 + 100:1024]


def test_read_file_feeds_queues_and_marks_eof(tmp_path):
    import queue
    f = tmp_path / 'in.raw'
    f.write_bytes(b'\x07' * (131072 + 10))
    q = queue.Queue()
    read_file.readFile(fs=1000, buffers=[q], inFile=str(f), dataOffset=4)
    items = []
    while not q.empty():
        items.append(q.get())
    # a regular file is handed over READ_BATCH chunks per item (whole chunks, stale tail included),
    # then the empty end-of-stream marker
    assert [len(i) for i in items] == [2 * 131072, 0]
    assert bytes(items[0][131072 + 6:131072 + 16]) == b'\x07' * 10      # stale tail of the chunk before (8-Q5)
    with pytest.raises(ValueError):
        read_file.readFile(fs=None, buffers=[q])


def test_cli_parser_matches_reference_options():
    from sdrterm_b200.sdrterm import buildParser, makeProcessor
    a = buildParser().parse_args(['-r', '1024k', '-c', '15k', '-w', '5k', '-d', '64', '--correct-iq',
                                  '-e', 'h', '-m', 'FM', '-X', '-i', 'x', '-o', 'y'])
    assert (a.fs, a.center, a.omegaOut, a.dec, a.correct_iq, a.enc, a.demod, a.swap) == \
        (1_024_000, 15000, 5000, 64, True, 'h', 'fm', True)
    info = file_util.parseRawType(None, a.fs, a.enc)
    p = makeProcessor(a, info)
    assert isinstance(p, dsp.DspProcessor) and p.demod == dem.fmDemod and p.decimatedFs == 16000
    b = buildParser().parse_args(['-r', '2400k', '-e', 'h', '--simo', '--vfos', '100000,-200000', '-d', '64',
                                  '--vfo-host', '127.0.0.1:0'])
    v = makeProcessor(b, file_util.parseRawType(None, b.fs, b.enc))
    assert isinstance(v, VfoProcessor) and v._nFreq == 3
    with pytest.raises(ValueError):
        makeProcessor(buildParser().parse_args(['-r', '1k', '-e', 'h', '-d', '1']), info)


def test_reference_import_names_resolve_to_this_build():
    sys.path.insert(0, os.path.join(ROOT, 'src'))
    try:
        import dsp.demodulation as d2
        import dsp.dsp_processor as p2
        import misc.read_file as r2
        import sdrterm as cli
        assert d2 is dem and p2 is dsp and r2 is read_file and callable(cli.main)
    finally:
        sys.path.remove(os.path.join(ROOT, 'src'))
        for k in [k for k in sys.modules if k in ('dsp', 'misc', 'sdrterm') or k.startswith(('dsp.', 'misc.'))]:
            del sys.modules[k]


def test_datatype_enum_and_from_wav():
    """file_util.py:46-97: the public types the reference's own test/misc/file_util_test.py imports."""
    from sdrterm_b200.misc.file_util import DataType, ExWaveFormat, WaveFormat
    from sdrterm_b200.misc.mappable_enum import MappableEnum
    assert [m.name for m in DataType] == list('bBhHiIfd')
    assert str(DataType.h) == 'h' and DataType['H'].value == np.dtype('=u2')
    assert DataType.dict()['f'] == np.dtype('=f4') and DataType.tuples()[0] == ('b', np.dtype('|i1'))
    assert MappableEnum.dict() == {} and MappableEnum.tuples() == ()
    fw = DataType.fromWav
    assert fw(8, WaveFormat.WAVE_FORMAT_PCM, None, False) == np.dtype('u1')
    assert fw(16, WaveFormat.WAVE_FORMAT_PCM, None, False) == np.dtype('<i2')
    assert fw(16, WaveFormat.WAVE_FORMAT_PCM, None, True) == np.dtype('>i2')
    assert fw(32, WaveFormat.WAVE_FORMAT_EXTENSIBLE, ExWaveFormat.PCM_U_BE, False) == np.dtype('>u4')
    assert fw(8, WaveFormat.WAVE_FORMAT_EXTENSIBLE, ExWaveFormat.PCM_S_LE, False) == np.dtype('i1')
    assert fw(64, WaveFormat.WAVE_FORMAT_IEEE_FLOAT, None, True) == np.dtype('>f8')
    for bad in ((24, WaveFormat.WAVE_FORMAT_PCM), (16, WaveFormat.WAVE_FORMAT_IEEE_FLOAT), (8, WaveFormat.WAVE_FORMAT_ALAW)):
        with pytest.raises(ValueError):
            fw(bad[0], bad[1], None, False)
    with pytest.raises(KeyError):
        file_util.checkWavHeader(None, 8000, 'q')
    with pytest.raises(TypeError):
        file_util.checkWavHeader(None, '2', 'B')


def test_repr_json_carries_the_keys_example_simo_scrapes():
    """example_simo.sh:96-118 greps "host", "vfos" (the CSV, not the array), "tunedFreq" and
    "decimatedFs" out of repr(processor) (dsp_processor.py:206-217 strips the 'Str' of vfosStr)."""
    import json
    p = VfoProcessor(2_400_000, vfoHost='localhost:9123', vfos='-100000,25000', center=-350000, tuned=155685000,
                     dec=64, omegaOut=5000, fileInfo={'bitsPerSample': np.dtype('>i2')})
    p.selectOutputFm()
    d = json.loads(repr(p))
    assert d['vfos'] == '-100000,25000,0' and 'vfosStr' not in d
    assert d['host'] == 'localhost' and d['port'] == 9123
    assert d['tunedFreq'] == 155685000 and d['decimatedFs'] == 2_400_000 // 64 and d['fs'] == 2_400_000
    assert d['encoding'] == '>i2' or d['encoding'] == 'int16' or 'i2' in d['encoding']
    q = dsp.DspProcessor(1_024_000, center=15000, dec=64, omegaOut=5000)
    dq = json.loads(repr(q))
    assert dq['centerFreq'] == 15000 and dq['decimatedFs'] == 16000


class _FakeEngine:
    made = []

    def __init__(self, plan, **kw):
        _FakeEngine.made.append(plan)

    def close(self):
        pass


def test_file_info_decides_dtype_and_byte_order_even_when_enc_is_passed(monkeypatch):
    """IOArgs hands the processor both -e and fileInfo (io_args.py:81-82,111-117); the reader uses
    fileInfo['bitsPerSample'] only (read_file.py:46-49): a WAV header overrides -e, host:port input
    is big-endian, -X flips whatever that is (ADVICE r1)."""
    import sdrterm_b200.engine as engine_mod
    monkeypatch.setattr(engine_mod, 'Engine', _FakeEngine)
    raw = bytes(131072)

    def plan_of(**kw):
        _FakeEngine.made.clear()
        p = dsp.DspProcessor(1_000_000, dec=64, omegaOut=5000, **kw)
        p.selectOutputFm()
        p._makeEngine(raw)
        return _FakeEngine.made[0]

    pl = plan_of(enc='B', fileInfo={'bitsPerSample': np.dtype('>i2')})
    assert pl.enc == 'h' and pl.swap is True
    pl = plan_of(enc='h', fileInfo={'bitsPerSample': np.dtype('>i2')}, swapEndianness=True)
    assert pl.enc == 'h' and pl.swap is False
    pl = plan_of(enc='d', fileInfo={'bitsPerSample': np.dtype('<f4')})
    assert pl.enc == 'f' and pl.swap is False
    pl = plan_of(enc='h', swapEndianness=True)
    assert pl.enc == 'h' and pl.swap is True
    pl = plan_of(fileInfo={'bitsPerSample': np.dtype('u1')}, swapEndianness=False)
    assert pl.enc == 'B' and pl.swap is False
    with pytest.raises(ValueError):
        plan_of()


def test_compiled_plugin_seam_is_importable_like_the_reference_expects():
    """read_file.py:58-63: `from dsp.fast.iq_correction import IQCorrection` must resolve."""
    src = os.path.join(ROOT, 'src')
    sys.path.insert(0, src)
    try:
        from dsp.fast.iq_correction import IQCorrection
    finally:
        sys.path.remove(src)
    c = IQCorrection(1_024_000)
    assert c.fs == 1_024_000 and c.impedance == 50 and c.inductance == 50 / 1_024_000
    c.impedance = 75
    c.fs = 2_400_000
    assert c.inductance == 75 / 2_400_000
    with pytest.raises(TypeError):
        c.correctIq(np.zeros(4, dtype=np.float64), np.zeros(1, dtype=np.complex128))


def test_reference_own_unit_tests_pass_against_the_shims(tmp_path):
    """The reference's API contract for this path: the cases of its test/dsp/dsp_processor_test.py
    and test/misc/{file_util,read_file,io_args,keyboard_interruptable_thread}_test.py, restated in
    tests/reference_unit_cases.py, run as the reference runs them: a fresh interpreter with
    PYTHONPATH=src, where ``dsp`` and ``misc`` are the shims."""
    import subprocess
    here = os.path.join(ROOT, 'tests')
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, 'src'))
    # rooted at tests/: collection never looks at directories above the checkout, which may be
    # unreadable
    r = subprocess.run([sys.executable, '-m', 'pytest', '-q', '-p', 'no:cacheprovider', '--rootdir', here,
                        '--basetemp', str(tmp_path / 'cases'), 'reference_unit_cases.py'],
                       env=env, cwd=here, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and ' passed' in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_cli_lifecycle_pid_file_and_signal(tmp_path):
    """src/sdrterm.py:172-231: `python -m sdrterm` writes a PID file, announces it, and a SIGTERM
    sets the halt flag -- both loops stop, the PID file is removed, exit status 0.  No input ever
    arrives on stdin here, so no device engine is created and this runs without a GPU."""
    import re
    import signal
    import subprocess
    import time
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, 'src'), TMPDIR=str(tmp_path))
    p = subprocess.Popen([sys.executable, '-m', 'sdrterm', '-r', '1024k', '-e', 'h', '-d', '64', '-w', '5k', '-vv'],
                         stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env,
                         cwd=str(tmp_path), text=True)
    lines = []
    deadline = time.time() + 60
    while time.time() < deadline:
        line = p.stderr.readline()
        lines.append(line)
        if 'decimatedFs' in line:                  # the repr JSON comes after the PID file line
            break
    head = ''.join(lines)
    m = re.search(r'PID file is created: (\S+)', head)
    assert m, head
    assert os.path.exists(m.group(1)) and open(m.group(1)).read().strip() == str(p.pid)
    assert f'Started proc Main: {p.pid}' in head
    time.sleep(0.5)
    p.send_signal(signal.SIGTERM)
    try:
        out, err = p.communicate(timeout=30)
    except subprocess.TimeoutExpired:
        p.kill()
        raise
    assert p.returncode == 0, err
    assert f'pid {p.pid} caught: SIGTERM' in err
    assert not os.path.exists(m.group(1))


def test_chunk_pool_reader_yields_views_with_the_same_bytes_and_stale_tail():
    """With a ChunkPool the reader fills pool buffers in place; chunk boundaries and the stale tail
    of a short final chunk (SURVEY 8-Q5) are what the copying reader produces."""
    data = bytes(range(256)) * 10 + b'\xee' * 100            # 2660 bytes, readSize 512, batch 2
    ref = [c.tobytes() for c in read_file.chunks(io.BytesIO(data), readSize=512, batch=2)]
    pool = read_file.ChunkPool(2, 1024)
    got = []
    for c in read_file.chunks(io.BytesIO(data), readSize=512, batch=2, pool=pool):
        home = pool.owner(c)
        assert home is not None and c.ctypes.data == home.ctypes.data      # a view, not a copy
        got.append(c.tobytes())
        pool.release(home)                                                  # what the consumer does
    assert got == ref
    assert pool.owner(np.zeros(8, dtype=np.uint8)) is None


class _RecordingEngine:
    """Stands in for the device: remembers what was submitted from where."""
    R, M = 1, 4

    class plan:
        big_endian_out = False

    def __init__(self):
        self.calls = []

    def submit(self, slot, raw_ptr, n, out_ptr):
        import ctypes
        self.calls.append((slot, raw_ptr, n, bytes((ctypes.c_uint8 * 16).from_address(raw_ptr))))

    def wait(self, slot):
        pass

    def close(self):
        pass


def test_consumer_sends_pool_buffers_in_place_and_hands_them_back(tmp_path):
    """File input through a ChunkPool: every batch is submitted from the pool buffer itself (no
    staging copy), in file order, and the buffer returns to the pool after the wait."""
    import queue
    import threading

    class Buf:
        def __init__(self, n):
            import ctypes
            self.u8 = np.zeros(n, dtype=np.uint8)
            self.ptr = ctypes.c_void_p(self.u8.ctypes.data)

        def view(self, dt):
            return self.u8.view(dt)

    eng = _RecordingEngine()

    class P(dsp.DspProcessor):
        def _makeEngine(self, c):
            self._chunkBytes = 131072
            return eng

        def _staging(self):
            self._hin = [Buf(self.MAX_BATCH * 131072) for _ in range(2)]
            self._hout = [Buf(self.MAX_BATCH * 4 * 8) for _ in range(2)]

    nchunks = 3 * read_file.READ_BATCH + 5
    f = tmp_path / 'in.raw'
    blob = np.arange(nchunks * 131072 // 4, dtype=np.uint32).view(np.uint8)
    f.write_bytes(blob.tobytes())
    pool = read_file.ChunkPool(2, read_file.READ_BATCH * 131072)
    homes = {r[0] for r in pool._ranges}
    p = P(1_000_000, dec=64, omegaOut=5000, enc='h')
    p.useInputPool(pool)
    q = queue.Queue()

    class Flag:
        value = 0
    th = threading.Thread(target=read_file.readFile, kwargs=dict(fs=1_000_000, buffers=[q], isDead=Flag(), inFile=str(f), pool=pool))
    th.start()
    with open(tmp_path / 'out.bin', 'wb') as out:
        p._processData(Flag(), q, out)
    th.join()
    assert [c[2] for c in eng.calls] == [read_file.READ_BATCH] * 3 + [5]
    assert all(c[1] in homes for c in eng.calls)                             # submitted in place
    assert [c[3] for c in eng.calls] == [blob[i * read_file.READ_BATCH * 131072:][:16].tobytes() for i in range(4)]
    assert [c[0] for c in eng.calls] == [0, 1, 0, 1]                         # alternating device slots
    assert pool._free.qsize() == 2                                           # every buffer came back
    assert '_inputPool' not in repr(p) and 'inputPool' not in p.__getstate__()
