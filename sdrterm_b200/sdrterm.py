"""``python -m sdrterm`` drop-in: same options as the reference's CLI (src/sdrterm.py:54-107) for
the demodulation path.  Plots are not part of this build (DESIGN.md 9).

A reader thread feeds raw chunks to the GPU consumer in this process; the reference's two-process
layout exists to overlap CPU work that no longer happens on the CPU."""
from __future__ import annotations

import argparse
import queue
import sys
import threading

from .misc.file_util import ENCODINGS, checkWavHeader, parseIntString
from .misc.read_file import readFile


class _Flag:
    """multiprocessing.Value-like stop flag."""

    def __init__(self):
        self.value = 0


def buildParser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog='sdrterm', description='B200 demodulation chain behind the sdrterm CLI')
    ap.add_argument('--fs', '-r', type=parseIntString, default=None, help='Sampling frequency in k/M/Samples per sec')
    ap.add_argument('--center-frequency', '-c', dest='center', type=parseIntString, default=0)
    ap.add_argument('--input', '-i', dest='inFile', default=None, help='file, host:port, or stdin')
    ap.add_argument('--output', '-o', dest='outFile', default=None, help='file or stdout')
    ap.add_argument('--plot', default=None, help='accepted and ignored (plots are out of scope)')
    ap.add_argument('--demodulation', '-m', dest='demod', type=str.lower, default='fm',
                    choices=['fm', 'nfm', 'am', 're', 'im', 'iq', 'usb', 'lsb'])
    ap.add_argument('--tuned-frequency', '-t', dest='tuned', type=parseIntString, default=0)
    ap.add_argument('--vfos', default=None, help='CSV of integer offsets from the tuned frequency')
    ap.add_argument('--decimation', '-d', dest='dec', type=int, default=2)
    ap.add_argument('--encoding', '-e', dest='enc', choices=list(ENCODINGS), default=None)
    ap.add_argument('--omega-out', '-w', dest='omegaOut', type=parseIntString, default=12500)
    ap.add_argument('--correct-iq', dest='correct_iq', action='store_true')
    ap.add_argument('--no-correct-iq', dest='correct_iq', action='store_false')
    ap.add_argument('--simo', action='store_true')
    ap.add_argument('--no-simo', dest='simo', action='store_false')
    ap.add_argument('--verbose', '-v', action='count', default=0)
    ap.add_argument('--smooth-output', dest='smooth_output', type=int, default=0)
    ap.add_argument('--vfo-host', dest='vfo_host', default='localhost')
    ap.add_argument('--swap-input-endianness', '-X', dest='swap', action='store_true')
    ap.add_argument('--seamless', dest='seamless', action='store_true',
                    help='not a reference option: filter and demodulate the whole stream as one signal '
                         'instead of each 131072-byte chunk (no transient at chunk edges; output '
                         'delayed by a few chunks; any -d; no --smooth-output)')
    ap.add_argument('--no-seamless', dest='seamless', action='store_false')
    ap.add_argument('--normalize-input', dest='normalize', action='store_true')
    ap.add_argument('--no-normalize-input', dest='normalize', action='store_false')
    return ap


def makeProcessor(a, fileInfo):
    """What IOArgs._initializeOutputHandlers does (src/misc/io_args.py:97-141)."""
    from .dsp.dsp_processor import DspProcessor
    from .dsp.vfo_processor import VfoProcessor
    if a.dec < 2:
        raise ValueError('Decimation must be at least 2.')
    kw = dict(center=a.center, omegaOut=a.omegaOut, tuned=a.tuned, dec=a.dec, smooth=a.smooth_output,
              fileInfo=fileInfo, swapEndianness=a.swap, correctIq=a.correct_iq, normalize=a.normalize)
    if a.seamless:
        kw['seamless'] = True
    fs = fileInfo['sampRate']
    proc = VfoProcessor(fs, vfoHost=a.vfo_host, vfos=a.vfos, **kw) if a.simo else DspProcessor(fs, **kw)
    {'fm': proc.selectOutputFm, 'nfm': proc.selectOutputFm, 'am': proc.selectOutputAm,
     're': proc.selectOutputReal, 'im': proc.selectOutputImag, 'iq': proc.selectOutputIq,
     'usb': proc.selectOutputUsb, 'lsb': proc.selectOutputLsb}[a.demod]()
    return proc


def _pidFile(pid: int):
    """PID file in the temp directory, announced on stderr (src/sdrterm.py:191-222); returns the
    function that removes it."""
    import os
    import re
    import tempfile
    import uuid
    from datetime import datetime, timezone
    from .misc.general_util import eprint, vprint
    iso = re.sub(r'[:\-+T]', '', datetime.now(timezone.utc).isoformat(timespec='seconds'))
    name = os.path.join(tempfile.gettempdir(), f'{iso}-sdrterm-{uuid.uuid4()}.pid')
    with open(name, 'w+') as fh:
        fh.write(str(pid) + '\n')
    eprint(f'PID file is created: {name}')

    def remove():
        try:
            os.unlink(name)
            vprint(f'PID file: {name} deleted')
        except OSError:
            pass
    return remove


def main(argv=None, lifecycle: bool = False) -> int:
    """``lifecycle``: install the reference's process lifecycle -- PID file, SIGINT/SIGTERM/... set
    the halt flag that both loops poll (src/sdrterm.py:172-231) -- as ``python -m sdrterm`` does;
    off when main() is called as a function (signal handlers belong to the main thread)."""
    import os
    from .misc import general_util as gu
    a = buildParser().parse_args(argv)
    if a.verbose > 1:
        gu.traceOn()
    elif a.verbose > 0:
        gu.verboseOn()
    isDead = _Flag()
    removePid = None
    if lifecycle:
        removePid = _pidFile(os.getpid())

        def stop():
            gu.tprint('Setting halt condition')
            isDead.value = 1
            removePid()
        gu.setSignalHandlers(os.getpid(), stop)
    fileInfo = checkWavHeader(a.inFile, a.fs, a.enc)           # a WAV header overrides -r / -e
    proc = makeProcessor(a, fileInfo)
    gu.tprint(f'Started proc Main: {os.getpid()}')
    print(repr(proc), file=sys.stderr, flush=True)          # unconditional: src/sdrterm.py:144
    buf = queue.Queue(maxsize=1024)
    pool = None
    if a.inFile and not fileInfo['isSocket'] and os.path.isfile(a.inFile):
        # a regular file is read READ_BATCH chunks at a time straight into page-locked buffers the
        # device then reads in place (no host copy between the page cache and the DMA)
        try:
            from ._native import PinnedBuffer
            from .misc.read_file import READ_BATCH, READ_SIZE, ChunkPool
            pool = ChunkPool(6, READ_BATCH * READ_SIZE, PinnedBuffer)
            proc.useInputPool(pool)
        except Exception:
            pool = None                                     # (no device: the engine will say so)
    def halt():
        isDead.value = 1

    from .misc.keyboard_interruptable_thread import KeyboardInterruptableThread
    rkw = dict(buffers=[buf], isDead=isDead, inFile=a.inFile, fs=fileInfo['sampRate'],
               dataOffset=fileInfo['dataOffset'], isSocket=fileInfo['isSocket'], pool=pool)
    # an exception in the reader (Ctrl-C included) sets the halt condition (src/sdrterm.py:195-231)
    reader = KeyboardInterruptableThread(halt, target=lambda: readFile(**rkw), name='reader', daemon=True)
    reader.start()
    try:
        proc.processData(isDead, buf, a.outFile)
    finally:
        isDead.value = 1
        if removePid is not None:
            removePid()
        gu.vprint('Main halted')
    return 0


if __name__ == '__main__':
    sys.exit(main(lifecycle=True))
