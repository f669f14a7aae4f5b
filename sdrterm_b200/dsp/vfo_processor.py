"""``VfoProcessor``: the ``--simo`` consumer (reference src/dsp/vfo_processor.py:36-126): rows =
the listed VFO offsets + the centre itself, one TCP client per row, big-endian doubles per row and
chunk.  The row math is one batched device call (every row is a CTA group of the same kernels)."""
from __future__ import annotations

import queue as _queue
import socket
import sys
from socketserver import BaseRequestHandler, TCPServer, ThreadingMixIn
from threading import Event, Thread

import numpy as np

from .dsp_processor import DspProcessor


def _free_port(host: str) -> int:
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind((host, 0))
        return s.getsockname()[1]


class _Server(ThreadingMixIn, TCPServer):
    allow_reuse_address = True
    daemon_threads = True


class VfoProcessor(DspProcessor):

    def __init__(self, fs, vfoHost: str = 'localhost', vfos: str | None = None, **kwargs):
        super().__init__(fs, **kwargs)
        if vfos is None or len(vfos) < 1:
            raise ValueError('simo mode cannot be used without the vfos option')
        self.vfosStr = vfos + ',0'
        offsets = [int(x) + self.centerFreq for x in vfos.split(',') if x is not None]
        offsets.append(self.centerFreq)                       # the centre is the last row (:45)
        self.vfos = np.array(offsets)
        self._nFreq = len(self.vfos)
        if ':' in vfoHost:
            self.host, port = vfoHost.split(':')
            self.port = int(port)
        else:
            self.host = vfoHost
            self.port = _free_port(self.host)
        self._clients = None
        self._rowQueue = None
        self._event = None

    def _rowsHz(self):
        return [int(v) for v in self.vfos]

    def _simo(self) -> bool:
        return True

    def _generateShift(self, c: int) -> None:
        """API parity (:71-78): the table itself, and the hand-out of one row per connected
        client; blocks until every row has a client."""
        w = -2j * np.pi * (self.vfos / self.fs)
        self._shift = np.exp(w[:, None] * np.arange(c)[None, :])
        if self._rowQueue is not None:
            for i in range(self._nFreq):
                self._rowQueue.put(i)
            self._rowQueue.join()
            # example_simo.sh waits for this line before it starts the stream (:165-170)
            print('Connection(s) established', file=sys.stderr, flush=True)

    def _emit(self, out: np.ndarray, noutputs: int, file) -> None:
        """Row r (``noutputs`` outputs) goes to client r; ``out`` rows already hold big-endian
        doubles (:84)."""
        if self._shift is None:
            self._generateShift(1)
        for r in range(self._nFreq):
            self._clients[r].write(out[r].tobytes())

    def processData(self, isDead, buffer, *args, **kwargs) -> None:
        self._rowQueue = _queue.Queue()
        self._event = Event()
        self._clients = {}
        outer = self

        class Handler(BaseRequestHandler):
            def handle(self):
                with self.request.makefile('wb', buffering=0) as fh:
                    row = outer._rowQueue.get()
                    outer._clients[row] = fh
                    outer._rowQueue.task_done()
                    outer._event.wait()

        with _Server((self.host, self.port), Handler) as server:
            th = Thread(target=server.serve_forever, daemon=True)
            try:
                print(f'\nAccepting connections on {server.socket.getsockname()}\n', file=sys.stderr, flush=True)
                th.start()
                self._processData(isDead, buffer)
            except KeyboardInterrupt:
                pass
            finally:
                self._event.set()
                self._isDead = True
                server.shutdown()
                th.join()
                if self._engine is not None:
                    self._engine.close()
                    self._engine = None

    def __getstate__(self):
        d = super().__getstate__()
        d['_clients'] = d['_rowQueue'] = d['_event'] = None
        return d
