"""``DspProcessor``: the reference's consumer object (src/dsp/dsp_processor.py:48-236) with the
same constructor, properties, selectors and ``processData`` contract, whose hot loop
(``_processChunk`` :140-149 + framing :162) runs on the GPU through one ``Engine`` handle.

Differences that matter to a caller:
  * chunks taken from the queue may be the reference's payload (1-D complex128 arrays, already
    decoded / normalised / IQ-corrected by the producer, read_file.py:100-112) **or** raw chunk
    bytes (``bytes`` / uint8 arrays), in which case decode, ``-X``, ``--normalize-input`` and
    ``--correct-iq`` also run on the device (keyword arguments ``enc``, ``swapEndianness``,
    ``normalize``, ``correctIq`` as misc/io_args.py passes them);
  * an empty chunk is a clean end of stream (SURVEY 8-Q7), ``-d`` values that do not divide the
    chunk produce ceil(N/q) outputs per chunk (8-Q1), ``re``/``im`` produce output (8-Q2);
  * no CUDA state exists before ``processData`` runs, so the object pickles into a spawned child
    exactly like the reference's (io_args.py:93).
"""
from __future__ import annotations

import queue as _queue
import sys
from sys import stdout
from typing import Any, Callable

import numpy as np

from .data_processor import DataProcessor
from .demodulation import amDemod, fmDemod, imagOutput, iqOutput, lsbDemod, realOutput, usbDemod

_DEMOD_NAME = {fmDemod: 'fm', amDemod: 'am', realOutput: 're', imagOutput: 'im', iqOutput: 'iq',
               usbDemod: 'usb', lsbDemod: 'lsb'}


def generateEllipFilter(fs: int, deg: int, Wn, btype: str):
    """Output low-pass design, SciPy's as in the reference (dsp_processor.py:39-45); design is
    setup, not hot path, and keeps the coefficients identical to the reference's.  The result is
    kept in the plan cache directory so that a command-line run that finds it does not import
    scipy.signal at all."""
    import os
    from ..plan import cache_dir
    root = cache_dir()
    path = os.path.join(root, f'ellip_{int(fs)}_{int(deg)}_{Wn!r}_{btype}.npy'.replace(os.sep, '_')) if root else None
    if path:
        try:
            return np.load(path)
        except Exception:
            pass
    from scipy.signal import ellip
    sos = ellip(deg, 1, 30, Wn, btype=btype, analog=False, output='sos', fs=fs)
    if path:
        try:
            os.makedirs(root, exist_ok=True)
            tmp = f'{path}.{os.getpid()}.tmp.npy'
            np.save(tmp, sos)
            os.replace(tmp, path)
        except OSError:
            pass
    return sos


class DspProcessor(DataProcessor):
    _FILTER_DEGREE = 3
    MAX_BATCH = 512         # chunks drained from the queue per device batch (64 MiB of raw input)
    _inputPool = None       # misc.read_file.ChunkPool shared with the reader (page-locked read buffers), see useInputPool

    def __init__(self, fs: int, center: int = 0, omegaOut: int = 0, tuned: int = 0, dec: int = 2,
                 smooth: bool = False, fileInfo: dict | None = None, **kwargs):
        self._demod = None
        self._shift = None
        self.bandwidth = None
        self.__fs = None
        self.__decimatedFs = None
        self._isDead = False
        self._outputFilters = []
        self._nFreq = 1
        self._decimationFactor = dec
        self.fs = fs
        self.centerFreq = center
        self.tunedFreq = tuned
        self.omegaOut = omegaOut
        self.smooth = smooth
        self.__fileInfo = fileInfo
        # ingest switches for raw-byte chunks (read_file.py:31-44 keyword names)
        self._enc = kwargs.get('enc')
        self._swap = bool(kwargs.get('swapEndianness', False))
        self._correctIq = bool(kwargs.get('correctIq', False))
        self._normalize = bool(kwargs.get('normalize', False))
        self._device = int(kwargs.get('device', 0))
        # seamless streaming (not a reference option, DESIGN.md section 11): the stream is filtered
        # and demodulated as one signal instead of chunk by chunk
        self._seamless = bool(kwargs.get('seamless', False))
        if self._seamless and smooth:
            raise ValueError('--smooth-output is per-chunk Savitzky-Golay by definition: not available with '
                             '--seamless')
        self._engine = None

    # ---------------------------------------------------------------- properties (:78-103)
    @property
    def fs(self) -> int:
        return self.__fs

    @fs.setter
    def fs(self, fs: int) -> None:
        self.__fs = fs
        self.__decimatedFs = fs // self._decimationFactor

    @property
    def decimation(self) -> int:
        return self._decimationFactor

    @decimation.setter
    def decimation(self, decimation: int) -> None:
        if decimation < 2:
            raise ValueError('Decimation must be at least 2.')
        self._decimationFactor = decimation
        self.fs = self.__fs

    @property
    def decimatedFs(self) -> int:
        return self.__decimatedFs

    # ---------------------------------------------------------------- demodulation choice (:105-138)
    def demod(self, *_, **__):
        pass

    def _setDemod(self, fun: Callable[[np.ndarray, np.ndarray], None], *filters) -> Callable[..., Any]:
        if fun is not None:
            self._outputFilters.clear()
            if len(filters):
                self._outputFilters.extend(*filters)
            setattr(self, 'demod', fun)
            return self.demod
        raise ValueError('Demodulation function, or filters not defined')

    def selectOutputFm(self):
        self.bandwidth = 12500
        self._setDemod(fmDemod, generateEllipFilter(self.__decimatedFs, self._FILTER_DEGREE,
                                                    self.omegaOut, 'lowpass'))

    def selectOutputAm(self):
        self.bandwidth = 10000
        self._setDemod(amDemod, generateEllipFilter(self.__decimatedFs, self._FILTER_DEGREE,
                                                    self.omegaOut, 'lowpass'))

    def selectOutputReal(self):
        self.bandwidth = self.decimatedFs
        self._setDemod(realOutput)

    def selectOutputImag(self):
        self.bandwidth = self.decimatedFs
        self._setDemod(imagOutput)

    def selectOutputIq(self):
        """Not a reference mode: the complex baseband itself, (Re, Im) doubles per output."""
        self.bandwidth = self.decimatedFs
        self._setDemod(iqOutput)

    def _checkSideband(self) -> None:
        if not 0 < self.omegaOut < self.__decimatedFs / 2:
            raise ValueError(f'usb/lsb: the sideband width -w {self.omegaOut} Hz must lie strictly between 0 and '
                             f'half the decimated rate ({self.__decimatedFs} / 2 Hz)')

    def selectOutputUsb(self):
        """Not a reference mode: the upper sideband [0, omegaOut] Hz from the tuned frequency as real
        audio (the band-pass ellip(3, 1, 30, omegaOut/2) moved up by omegaOut/2)."""
        self._checkSideband()
        self.bandwidth = self.omegaOut
        self._setDemod(usbDemod, generateEllipFilter(self.__decimatedFs, self._FILTER_DEGREE,
                                                     self.omegaOut / 2, 'lowpass'))

    def selectOutputLsb(self):
        """Not a reference mode: the lower sideband [-omegaOut, 0] Hz, as selectOutputUsb."""
        self._checkSideband()
        self.bandwidth = self.omegaOut
        self._setDemod(lsbDemod, generateEllipFilter(self.__decimatedFs, self._FILTER_DEGREE,
                                                     self.omegaOut / 2, 'lowpass'))

    # ---------------------------------------------------------------- NCO table (:185-187)
    def _generateShift(self, c: int) -> None:
        """Kept for API parity (tests read ``_shift``); the device path builds its own phasor
        tables from the same expression (plan.py: reference_w)."""
        if self.centerFreq:
            self._shift = np.array([np.exp(-2j * np.pi * (self.centerFreq / self.__fs) * np.arange(c))])

    # ---------------------------------------------------------------- device engine
    def _rowsHz(self) -> list[int]:
        return [int(self.centerFreq)]

    def _simo(self) -> bool:
        return False

    def _demodName(self) -> str:
        name = _DEMOD_NAME.get(getattr(self, 'demod', None))
        if name is None:
            raise ValueError('no demodulation selected (call selectOutputFm/Am/Real/Imag/Iq/Usb/Lsb first)')
        return name

    def _makeEngine(self, first):
        from ..engine import Engine
        from ..plan import cached_plan
        if isinstance(first, np.ndarray) and np.iscomplexobj(first):
            enc, swap, ciq, norm = 'Z', False, False, False       # producer already did these
            chunk_bytes = first.size * 16
        else:
            # the header (or host:port => network order) decides dtype and byte order whenever
            # fileInfo is present, exactly as the reference's reader does (read_file.py:46-49 uses
            # fileInfo['bitsPerSample'], never -e); -X flips whatever order that is
            swap = self._swap
            if self.__fileInfo is not None:
                dt = np.dtype(self.__fileInfo['bitsPerSample'])
                enc = dt.char
                big = dt.byteorder == '>' or (dt.byteorder == '=' and sys.byteorder == 'big')
                swap = bool(swap) ^ bool(big and dt.itemsize > 1)
            else:
                enc = self._enc
            if enc is None:
                raise ValueError('raw chunks need the sample encoding (enc=... or fileInfo)')
            ciq, norm = self._correctIq, self._normalize
            nb = len(first) if not isinstance(first, np.ndarray) else first.nbytes
            chunk_bytes = 131072 if nb % 131072 == 0 else nb     # the reader may hand over several chunks at once
        plan, tc = cached_plan(self.__fs, enc, self._decimationFactor, self._rowsHz(), simo=self._simo(),
                               swap=swap, correct_iq=ciq, normalize=norm, demod=self._demodName(),
                               omega_out=self.omegaOut, chunk_bytes=chunk_bytes,
                               **({'seamless': True} if self._seamless else {}))
        self._chunkBytes = chunk_bytes
        # --smooth-output (dsp_processor.py:159-160): standard mode only, the SIMO override of
        # _transformData never smooths (vfo_processor.py:80-84)
        smooth = int(self.smooth) if (self.smooth and not self._simo()) else 0
        return Engine(plan, max_chunks=self.MAX_BATCH, device=self._device, smooth=smooth, tc=tc)

    def _rowDoubles(self) -> int:
        """Doubles per chunk and row of the engine's output: 2M for iq ((Re, Im) pairs), M otherwise."""
        return 2 * self._engine.M if self.demod is iqOutput else self._engine.M

    @staticmethod
    def _asBytes(chunk) -> np.ndarray:
        if isinstance(chunk, np.ndarray):
            if np.iscomplexobj(chunk):
                chunk = np.ascontiguousarray(chunk, dtype=np.complex128)
            return np.ascontiguousarray(chunk).view(np.uint8).reshape(-1)
        return np.frombuffer(chunk, dtype=np.uint8)

    def _emit(self, out: np.ndarray, nchunks: int, file) -> None:
        """Standard mode: one stream, native doubles, chunk after chunk (:162)."""
        file.write(out[0].tobytes())

    def _staging(self):
        """Two page-locked host buffers each way (cudaHostAlloc through the C ABI)."""
        from .._native import PinnedBuffer
        eng = self._engine
        n = self.MAX_BATCH
        self._hin = [PinnedBuffer(n * self._chunkBytes) for _ in range(2)]
        self._hout = [PinnedBuffer(eng.R * n * self._rowDoubles() * 8) for _ in range(2)]

    def _processData(self, isDead, buffer, file=None) -> None:
        """The consumer loop (dsp_processor.py:164-183), double-buffered: while the device works on
        batch i (H2D, kernels, D2H on the slot's stream: sdrb_submit), the host drains the queue
        into the other pinned buffer and frames / writes the output of batch i-1 (sdrb_wait).
        A batch is whatever the queue holds (at most MAX_BATCH chunks), so a live stream is not
        held back waiting for a full batch."""
        if self._seamless:
            return self._processSeamless(isDead, buffer, file)
        eof = False
        pending = None                                   # (slot, nchunks) in flight
        b = 0
        while not (self._isDead or isDead.value or eof):
            first = self._next(isDead, buffer)
            if first is None:                            # halted while waiting for input
                break
            batch = [first]
            have = self._itemChunks(first)
            while have < self.MAX_BATCH:
                try:
                    batch.append(buffer.get_nowait())
                except _queue.Empty:
                    break
                have += self._itemChunks(batch[-1])
            chunks = []
            nch = 0
            pool = self._inputPool
            for c in batch:
                if c is None or len(c) == 0:          # end-of-stream marker (read_file.py:169-171)
                    eof = True
                    break
                if self._engine is None:
                    self._engine = self._makeEngine(c)
                    self._staging()
                a = self._asBytes(c)                   # one chunk, or several whole chunks read at once
                if a.size % self._chunkBytes:
                    raise ValueError('queue items must be whole chunks of the size of the first one')
                home = pool.owner(a) if pool is not None else None
                if home is not None and a.size // self._chunkBytes <= self.MAX_BATCH:
                    # the reader filled a page-locked pool buffer: the device reads it where it
                    # lies (the staged chunks before it go first, in order)
                    pending, b = self._flush(chunks, pending, b, file)
                    chunks = []
                    slot = b & 1
                    n = a.size // self._chunkBytes
                    self._engine.submit(slot, a.ctypes.data, n, self._hout[slot].ptr.value)
                    if pending is not None:
                        self._drain(pending, file)
                    pending = (slot, n, home)
                    b += 1
                    continue
                chunks.append(a)
                nch += a.size // self._chunkBytes
            pending, b = self._flush(chunks, pending, b, file)
        if pending is not None:
            self._drain(pending, file)

    def _flush(self, flat, pending, b, file):
        """Copy the collected chunks into the pinned staging buffers, MAX_BATCH at a time, and
        submit them (a batch of multi-chunk items may exceed MAX_BATCH: split it)."""
        pos = 0
        while flat:
            slot = b & 1
            hin = self._hin[slot].u8
            n = 0
            while flat and n < self.MAX_BATCH:
                a = flat[0]
                take = min(a.size // self._chunkBytes - pos, self.MAX_BATCH - n)
                hin[n * self._chunkBytes:(n + take) * self._chunkBytes] = \
                    a[pos * self._chunkBytes:(pos + take) * self._chunkBytes]
                n += take
                pos += take
                if pos * self._chunkBytes == a.size:
                    flat.pop(0)
                    pos = 0
            self._engine.submit(slot, self._hin[slot].ptr.value, n, self._hout[slot].ptr.value)
            if pending is not None:
                self._drain(pending, file)
            pending = (slot, n, None)
            b += 1
        return pending, b

    def _processSeamless(self, isDead, buffer, file) -> None:
        """The consumer loop of the seamless mode, synchronous: every batch goes through
        ``Engine.stream`` (which emits the chunks that have become final), and at end of stream or on
        halt ``Engine.stream_end`` emits the chunks still held back, so no tail is lost."""
        eof = False
        pool = self._inputPool
        while not (self._isDead or isDead.value or eof):
            first = self._next(isDead, buffer)
            if first is None:
                break
            batch = [first]
            have = self._itemChunks(first)
            while have < self.MAX_BATCH:
                try:
                    batch.append(buffer.get_nowait())
                except _queue.Empty:
                    break
                have += self._itemChunks(batch[-1])
            for c in batch:
                if c is None or len(c) == 0:
                    eof = True
                    break
                if self._engine is None:
                    self._engine = self._makeEngine(c)
                a = self._asBytes(c)
                if a.size % self._chunkBytes:
                    raise ValueError('queue items must be whole chunks of the size of the first one')
                out = self._engine.stream(a)
                home = pool.owner(a) if pool is not None else None
                if home is not None:
                    pool.release(home)                   # stream() has copied the bytes to the device
                if out.shape[1]:
                    self._emit(out, out.shape[1] // self._rowDoubles(), file)
        if self._engine is not None:
            out = self._engine.stream_end()
            if out.shape[1]:
                self._emit(out, out.shape[1] // self._rowDoubles(), file)

    def useInputPool(self, pool) -> None:
        """Queue items that are views of ``pool``'s buffers (misc.read_file.ChunkPool) are sent to
        the device from where they lie and handed back to the pool afterwards."""
        self._inputPool = pool

    @staticmethod
    def _itemChunks(c) -> int:
        """Chunks a queue item holds (1 for the reference's complex payload or a single raw chunk)."""
        if c is None or isinstance(c, np.ndarray) and np.iscomplexobj(c):
            return 1
        nb = c.nbytes if isinstance(c, np.ndarray) else len(c)
        return max(1, nb // 131072)

    def _next(self, isDead, buffer):
        """Blocking ``buffer.get()`` that still notices the halt flag (the reference's consumer is
        a process that dies with the signal; this one may be a thread)."""
        while True:
            try:
                return buffer.get(timeout=0.25)
            except _queue.Empty:
                if self._isDead or isDead.value:
                    return None

    def _drain(self, pending, file) -> None:
        slot, n, home = pending
        eng = self._engine
        eng.wait(slot)
        if home is not None:
            self._inputPool.release(home)                 # the device has the bytes: the reader may refill it
        W = self._rowDoubles()
        out = self._hout[slot].view(np.float64)[:eng.R * n * W].reshape(eng.R, n * W)
        if eng.plan.big_endian_out:
            out = out.view('>f8')
        self._emit(out, n, file)

    def processData(self, isDead, buffer, f: str | None, *args, **kwargs) -> None:
        with open(f, 'wb') if f is not None else open(stdout.fileno(), 'wb', closefd=False) as file:
            try:
                self._processData(isDead, buffer, file)
                file.flush()
            except KeyboardInterrupt:
                pass
            finally:
                if self._engine is not None:
                    self._engine.close()
                    self._engine = None
                for m in ('close', 'join_thread'):
                    if hasattr(buffer, m):
                        getattr(buffer, m)()

    # ---------------------------------------------------------------- pickling / repr
    def __getstate__(self):
        d = dict(self.__dict__)
        d['_engine'] = None
        d.pop('_hin', None), d.pop('_hout', None), d.pop('_inputPool', None)
        return d

    def __repr__(self):
        from json import dumps
        # keys lose a trailing 'Str' (vfosStr -> "vfos", the CSV example_simo.sh scrapes; the array
        # of the same name is skipped), dsp_processor.py:206-217
        d = {(k[:-3] if 'Str' in k else k): v for k, v in self.__dict__.items()
             if not (v is None or k.startswith('_') or callable(v) or isinstance(v, np.ndarray))}
        if self.__fileInfo is not None:
            d['encoding'] = str(self.__fileInfo.get('bitsPerSample'))
        d['fs'] = self.__fs
        d['decimatedFs'] = self.__decimatedFs
        if self._seamless:
            d['seamless'] = True
        name = _DEMOD_NAME.get(getattr(self, 'demod', None))
        if name in ('usb', 'lsb'):
            d['demodulation'] = name
        return dumps(d, indent=2, default=str)

    def __str__(self):
        return self.__class__.__name__
