"""The original sdrterm project's unit tests for this path, restated: the cases of its
test/dsp/dsp_processor_test.py, test/misc/file_util_test.py, test/misc/read_file_test.py,
test/misc/io_args_test.py and test/misc/keyboard_interruptable_thread_test.py (SURVEY.md section 4),
written against that project's top-level import names (``dsp.*``, ``misc.*``).

The suite does not collect this file itself: tests/test_host_api.py runs it in a fresh interpreter
with PYTHONPATH=src, so those names resolve to this build through the ``src/`` shims, as they
resolve to the original packages in the original project's own test run."""
import math
import struct
import threading

import numpy as np
import pytest

import dsp.demodulation as dem
from dsp.data_processor import DataProcessor
from dsp.dsp_processor import DspProcessor
from dsp.vfo_processor import VfoProcessor
from misc.file_util import DataType, checkWavHeader
from misc.io_args import IOArgs
from misc.keyboard_interruptable_thread import KeyboardInterruptableThread
from misc.mappable_enum import MappableEnum
from misc.read_file import generateDomain, readFile


# ------------------------------------------------------------------ test/dsp/dsp_processor_test.py
FS, CENTER, NSHIFT, DEC = 48000, -1000, 8, 3


def test_processor_properties_and_demod_selection():
    p = DspProcessor(FS, omegaOut=250)
    assert p.fs == FS
    p.selectOutputFm()
    assert p.demod == dem.fmDemod                 # the module's function object itself
    p.selectOutputAm()
    assert p.demod == dem.amDemod
    with pytest.raises(ValueError):
        p.decimation = 1
    with pytest.raises(AttributeError):
        p.decimatedFs = 1
    p.decimation = DEC
    assert p.decimation == DEC and p.decimatedFs == FS / DEC


def test_set_demod_rejects_missing_or_uncallable():
    p = DspProcessor(FS)
    with pytest.raises(ValueError):
        p._setDemod(None, ())
    with pytest.raises(TypeError):
        p._setDemod('asdf', None)


def test_generate_shift_is_none_at_centre_zero_and_exact_otherwise():
    p = DspProcessor(FS)
    p._generateShift(NSHIFT)
    assert p._shift is None
    p.centerFreq = CENTER
    p._generateShift(NSHIFT)
    for k in range(NSHIFT):
        assert p._shift[0][k] == np.pow(math.e, -2j * math.pi * (CENTER / FS) * k)


def test_process_data_argument_errors_and_abstract_base():
    p = DspProcessor(FS)
    with pytest.raises(FileNotFoundError):
        p.processData(None, None, '')
    with pytest.raises(AttributeError):
        p.processData(None, None, None)
    with pytest.raises(TypeError):
        DataProcessor()


# ------------------------------------------------------------------ test/misc/file_util_test.py
_GUID_TAIL = b'\x00\x00\x00\x00\x10\x00\x80\x00\x00\xAA\x00\x38\x9B\x71'


def _header(tag=b'RIFF', fmt=1, bits=16, nch=2, rate=8000, sub=None, guid=_GUID_TAIL, wave=b'WAVE',
            fmt_tag=b'fmt ', data=b'data'):
    e = '>' if tag == b'RIFX' else '<'
    align = nch * bits // 8
    body = struct.pack(e + 'HHIIHH', fmt, nch, rate, rate * align, align, bits)
    if sub is not None:                           # WAVE_FORMAT_EXTENSIBLE: cbSize, valid bits, mask, GUID
        body += struct.pack(e + 'HHIH', 22, bits, 3, sub) + guid
    fmt_chunk = fmt_tag + struct.pack(e + 'I', len(body)) + body
    payload = b'\0' * 64
    rest = wave + fmt_chunk + data + struct.pack(e + 'I', len(payload)) + payload
    return tag + struct.pack(e + 'I', len(rest)) + rest


@pytest.mark.parametrize('head, dtype', [
    (_header(fmt=1, bits=8), 'u1'),
    (_header(fmt=1, bits=16), '<i2'),
    (_header(fmt=0xFFFE, bits=32, sub=0x01), '<i4'),
    (_header(fmt=3, bits=32), '<f4'),
    (_header(fmt=3, bits=64), '<f8'),
    (_header(tag=b'RIFX', fmt=1, bits=16), '>i2'),
    (_header(fmt=1, bits=16, nch=1), '<i2'),
])
def test_valid_wav_headers(tmp_path, head, dtype):
    f = tmp_path / 'in.wav'
    f.write_bytes(head)
    info = checkWavHeader(str(f), None, None)
    assert info['bitsPerSample'] == np.dtype(dtype) and info['sampRate'] == 8000 and not info['isSocket']


@pytest.mark.parametrize('head', [
    b'RIFZ' + _header()[4:],                      # neither RIFF nor RIFX
    b'XXXX' + _header()[4:],                      # no RIFF tag in a .wav
    _header(wave=b'WAVX'),
    _header(fmt_tag=b'fmtX'),
    _header(fmt=1, bits=24),                      # PCM width without a dtype
    _header(fmt=3, bits=16),                      # half floats
    _header(fmt=6, bits=8),                       # A-law
    _header(fmt=0xFFFE, bits=16, sub=0x01, guid=b'\1' * 14),
    _header(data=b'atad'),                        # no data section
])
def test_malformed_wav_headers(tmp_path, head):
    f = tmp_path / 'in.wav'
    f.write_bytes(head)
    with pytest.raises(ValueError):
        checkWavHeader(str(f), None, None)


def test_raw_input_needs_rate_and_encoding(tmp_path):
    f = tmp_path / 'in.raw'
    f.write_bytes(b'\0' * 64)
    info = checkWavHeader(str(f), 8000, 'h')
    assert info['bitsPerSample'] == DataType.h.value and info['sampRate'] == 8000 and info['dataOffset'] == 0
    with pytest.raises(ValueError):
        checkWavHeader(str(f), None, 'h')
    with pytest.raises(ValueError):
        checkWavHeader(str(f), 8000, None)
    with pytest.raises(KeyError):
        checkWavHeader(None, 8000, 'q')


def test_mappable_enum_lists_its_members():
    assert MappableEnum.dict() == {} and MappableEnum.tuples() == ()
    assert DataType.dict()['B'] == np.dtype('u1') and [k for k, _ in DataType.tuples()] == list('bBhHiIfd')


# ------------------------------------------------------------------ test/misc/read_file_test.py
def test_generate_domain():
    assert generateDomain('B') == (0, 1 / 255)
    assert generateDomain('b') == (-128, 1 / 255)
    assert generateDomain('h') == (-32768, 1 / 65535)
    assert generateDomain('H') == (0, 1 / 65536)
    assert generateDomain('i') == (-2147483648, 1 / 4294967295)
    assert generateDomain('I') == (0, 1 / 4294967295)
    assert generateDomain('f') is None and generateDomain('d') is None


def test_read_file_needs_a_rate():
    with pytest.raises(ValueError):
        readFile()


# ------------------------------------------------------------------ test/misc/io_args_test.py
@pytest.mark.parametrize('simo, kind', [(True, VfoProcessor), (False, DspProcessor)])
def test_output_handlers_build_the_processor_and_its_process(simo, kind):
    IOArgs.strct = {}
    processes, buffers = [], []
    kw = dict(vfos='-100000,100000', vfoHost='127.0.0.1:0') if simo else {}
    IOArgs._initializeOutputHandlers(isDead=None, fs=2_400_000, dm='fm', outFile=None, simo=simo, pl=None,
                                     processes=processes, buffers=buffers, dec=64, omegaOut=5000, **kw)
    p = IOArgs.strct['processor']
    assert type(p) is kind and p.demod == dem.fmDemod
    assert len(processes) == 1 and len(buffers) == 1 and not processes[0].is_alive()
    with pytest.raises(ValueError):
        IOArgs._initializeOutputHandlers(isDead=None, fs=2_400_000, dm='xx', simo=False, processes=[], buffers=[])


# ------------------------------------------------------------------ test/misc/keyboard_interruptable_thread_test.py
def test_thread_needs_a_shutdown_hook():
    with pytest.raises(ValueError):
        KeyboardInterruptableThread(None, target=lambda: None)


@pytest.mark.parametrize('exc', [KeyboardInterrupt, RuntimeError])
def test_uncaught_exception_runs_the_shutdown_hook(exc):
    saved = threading.excepthook
    called = []

    def target():
        raise exc('stop')
    try:
        t = KeyboardInterruptableThread(lambda: called.append(True), target=target)
        t.start()
        t.join(10)
        assert not t.is_alive() and called == [True]
    finally:
        threading.excepthook = saved
