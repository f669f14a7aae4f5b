"""Engine: one libsdrterm_b200 handle built from a Plan (sdrterm_b200/plan.py).

This is the thin host layer between the reference-shaped processors (dsp/*.py) and the C ABI.
Inputs are whole 131072-byte chunks of raw IQ bytes; outputs are float64 rows
``[row][chunk][W]`` framed as the reference frames them (native doubles, or big-endian in SIMO).
W is M, except for iq output: 2M doubles, (Re, Im) of each decimator output interleaved
(usb / lsb: M real doubles of single-sideband audio).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat
from .plan import Plan, build_tc_or_none


def _dp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Engine:
    def __init__(self, plan: Plan, max_chunks: int = 256, device: int = 0, use_tc: bool = True,
                 keep_decimated: bool = False, keep_x0: bool = False, smooth: int = 0, tc='build'):
        self.plan = plan
        self.max_chunks = int(max_chunks)
        self.device = int(device)
        self._h = C.c_void_p()
        self._keep = []
        L = nat.lib()
        pl = plan
        cfg = nat.Config()
        cfg.abi_version = nat.ABI_VERSION
        cfg.device = self.device
        cfg.enc = pl.enc.encode()
        cfg.swap = int(pl.swap)
        cfg.correct_iq = int(pl.correct_iq)
        cfg.normalize = int(pl.norm is not None)
        cfg.demod = nat.DEMOD_CODE[pl.demod]
        cfg.big_endian_out = int(pl.big_endian_out)
        cfg.q, cfg.N, cfg.edge, cfg.R = pl.q, pl.N, pl.edge, pl.R
        cfg.n_out_sections = 0 if pl.out_sos is None else pl.out_sos.shape[0]
        cfg.max_chunks = self.max_chunks
        cfg.iq_L = pl.Liq
        cfg.norm_xmin, cfg.norm_k = pl.norm if pl.norm is not None else (0.0, 0.0)
        self.seamless = bool(getattr(pl, 'seamless', False))
        cfg.seamless = int(self.seamless)
        if pl.demod == 'iq' and smooth:
            raise ValueError('--smooth-output is not available with iq output')
        if self.seamless and smooth:
            raise ValueError('--smooth-output is per-chunk Savitzky-Golay by definition: not available in '
                             'seamless mode')
        tab = nat.Tables()

        def put(name, arr):
            a = np.ascontiguousarray(arr)
            if a.dtype == np.complex128:
                a = a.view(np.float64)
            a = np.ascontiguousarray(a, dtype=np.float64)
            self._keep.append(a)
            setattr(tab, name, _dp(a))

        m = pl.modes
        for name, arr in (('p', m.p), ('P', pl.P), ('rho', m.rho), ('rho_p', m.rho_p), ('c', m.c),
                          ('zhat', m.zhat), ('xi', m.xi), ('Ec', pl.Ec), ('Oc', pl.Oc),
                          ('Ppow', pl.Ppow), ('pk', pl.Pk), ('Pt', pl.Pt), ('bx', pl.bx), ('bnd', pl.bnd), ('lam_j', pl.lam_j),
                          ('lam_k', pl.lam_k), ('mu_k', pl.mu_k), ('T2', pl.T2),
                          ('T3', pl.T3), ('T1', pl.T1), ('Ehead', pl.Ehead), ('Eend', pl.Eend),
                          ('alpha', pl.alpha), ('alphaT', pl.alphaT), ('beta', pl.beta),
                          ('betaT', pl.betaT), ('gamma', pl.gamma), ('phE', pl.phE), ('psiY', pl.psiY)):
            put(name, arr)
        put('out_sos', pl.out_sos if pl.out_sos is not None else np.zeros(6))
        tab.g0, tab.d, tab.k_bnd = m.g0, m.d, int(pl.k_bnd)
        tab.lam, tab.lam_q, tab.lam_inv = pl.lam, pl.lam_q, pl.lam_inv
        tab.RL = int(pl.RL)
        for i in range(8):
            tab.run_len[i] = int(pl.run_len[i])
            tab.lam_run[i] = float(pl.lam_run[i])
        nco = np.ascontiguousarray(pl.use_nco, dtype=np.uint8)
        self._keep.append(nco)
        tab.use_nco = nco.ctypes.data_as(C.POINTER(C.c_uint8))
        tab.sos_Lseg = int(pl.sos_Lseg)
        if pl.sos_CA is not None:
            put('sos_CA', pl.sos_CA)
            put('sos_AP', pl.sos_AP)
        tab.lam_N = float(pl.lam_N)
        tab.lam_tile[0], tab.lam_tile[1] = float(pl.lam_tile[0]), float(pl.lam_tile[1])
        if pl.fm_interp is not None:
            put('fm_interp', pl.fm_interp)
        if getattr(pl, 'ssb_rot', None) is not None:
            tab.ssb_omega = float(pl.ssb_omega)
            put('ssb_rot', pl.ssb_rot)
        if self.seamless:
            tab.lookahead, tab.fs = int(pl.lookahead), int(pl.fs)
            step = np.ascontiguousarray(pl.chunk_step, dtype=np.int64)
            self._keep.append(step)
            tab.chunk_step = step.ctypes.data_as(C.POINTER(C.c_int64))
            put('PN', pl.PN)
            if pl.sos_AM is not None:
                put('sos_AM', pl.sos_AM)
                put('sos_CAM', pl.sos_CAM)
        # tc: prebuilt tensor-core tables (plan.cached_plan), or 'build'
        self.tc = (build_tc_or_none(pl) if isinstance(tc, str) else tc) if use_tc else None
        if self.tc is not None:
            tc = self.tc
            tab.tc_enable, tab.tc_K, tab.tc_isz = 1, tc.K, tc.isz
            tab.tc_ncol, tab.tc_nout, tab.tc_npad, tab.tc_S = tc.NCOL, tc.nout, tc.Npad, tc.S
            tab.tc_S_yl, tab.tc_nrowc, tab.tc_a_signed = tc.S_yl, tc.rowc.shape[1], int(tc.a_signed)
            put('tc_rowc', tc.rowc)
            bq = np.ascontiguousarray(tc.Bq, dtype=np.int8)
            self._keep.append(bq)
            tab.tc_Bq = bq.ctypes.data_as(C.POINTER(C.c_int8))
            put('tc_cst', tc.cst)
            for i in range(16):
                tab.tc_xor[i] = int(tc.xor_mask[i])
        nat.check(L.sdrb_create(C.byref(cfg), C.byref(tab), C.byref(self._h)))
        self.M = int(L.sdrb_outputs_per_chunk(self._h))
        self.W = int(L.sdrb_row_doubles(self._h))       # doubles per chunk and row of the output
        if keep_decimated:
            nat.check(L.sdrb_keep_decimated(self._h, 1), self._h)
        if keep_x0:
            nat.check(L.sdrb_keep_x0(self._h, 1), self._h)
        if smooth:
            self.set_smooth(int(smooth))
        self.chunk_bytes = int(L.sdrb_chunk_bytes(self._h))
        self.R = pl.R

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if self._h:
            nat.lib().sdrb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ hot path
    def _nchunks(self, nbytes: int) -> int:
        n, r = divmod(nbytes, self.chunk_bytes)
        if r:
            raise ValueError(f'input of {nbytes} bytes is not a whole number of '
                             f'{self.chunk_bytes}-byte chunks')
        return n

    def process(self, raw, out: np.ndarray | None = None) -> np.ndarray:
        """Host bytes in, (R, nchunks*W) float64 out (H2D + kernels + D2H, synchronous).  With
        big-endian framing the returned array holds the byte-swapped doubles (dtype '>f8')."""
        buf = np.frombuffer(raw, dtype=np.uint8) if not isinstance(raw, np.ndarray) else raw
        buf = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        n = self._nchunks(buf.size)
        if self.seamless:
            raise nat.SdrbError('seamless engine: use stream() / stream_end()')
        dt = np.dtype('>f8') if self.plan.big_endian_out else np.dtype('=f8')
        if out is None:
            out = np.empty((self.R, n * self.W), dtype=dt)
        if n:
            nat.check(nat.lib().sdrb_process(self._h, buf.ctypes.data, n, out.ctypes.data), self._h)
        return out

    # ------------------------------------------------------------------ seamless streaming
    @property
    def lookahead(self) -> int:
        """D: in seamless mode a chunk's output is final once the D chunks after it exist."""
        return int(nat.lib().sdrb_stream_lookahead(self._h)) if self.seamless else 0

    def _out_array(self, nchunks: int) -> np.ndarray:
        dt = np.dtype('>f8') if self.plan.big_endian_out else np.dtype('=f8')
        return np.empty(self.R * nchunks * self.W, dtype=dt)

    def _rows(self, flat: np.ndarray, k: int) -> np.ndarray:
        return flat[:self.R * k * self.W].reshape(self.R, k * self.W)

    def stream(self, raw) -> np.ndarray:
        """Seamless mode: take whole chunks of the stream, return (R, k*W) for the k chunks that have
        become final (the stream is filtered as one signal; see DESIGN.md section 11).  Batches
        larger than ``max_chunks`` are fed in pieces."""
        if not self.seamless:
            raise nat.SdrbError('stream() needs a plan built with seamless=True')
        buf = np.frombuffer(raw, dtype=np.uint8) if not isinstance(raw, np.ndarray) else raw
        buf = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        n = self._nchunks(buf.size)
        parts = []
        for c0 in range(0, n, self.max_chunks):
            k = min(self.max_chunks, n - c0)
            out = self._out_array(k + self.lookahead)
            got = C.c_size_t(0)
            nat.check(nat.lib().sdrb_stream(self._h, buf[c0 * self.chunk_bytes:].ctypes.data, k, out.ctypes.data,
                                            C.byref(got)), self._h)
            parts.append(self._rows(out, got.value))
        if not parts:
            return self._rows(self._out_array(0), 0)
        return np.concatenate(parts, axis=1) if len(parts) > 1 else parts[0]

    def stream_end(self) -> np.ndarray:
        """Seamless mode: end of stream.  Returns the chunks still held back, filtered with the stream's
        real end as the boundary, and resets the stream (IQ corrector included)."""
        if not self.seamless:
            raise nat.SdrbError('stream_end() needs a plan built with seamless=True')
        out = self._out_array(max(1, self.lookahead))
        got = C.c_size_t(0)
        nat.check(nat.lib().sdrb_stream_end(self._h, out.ctypes.data, C.byref(got)), self._h)
        return self._rows(out, got.value)

    def stream_device(self, raw_ptr: int, nchunks: int, out_ptr: int, stream: int = 0) -> int:
        """Device pointers in/out, only enqueued on ``stream``; returns the number of chunks emitted."""
        got = C.c_size_t(0)
        nat.check(nat.lib().sdrb_stream_device(self._h, raw_ptr, nchunks, out_ptr, stream, C.byref(got)), self._h)
        return got.value

    def stream_end_device(self, out_ptr: int, stream: int = 0) -> int:
        got = C.c_size_t(0)
        nat.check(nat.lib().sdrb_stream_end_device(self._h, out_ptr, stream, C.byref(got)), self._h)
        return got.value

    def set_smooth(self, window: int, polyorder: int = 3) -> None:
        """``--smooth-output``: ``scipy.signal.savgol_filter(z, window, 3)`` on every chunk's output
        row (reference dsp_processor.py:159-160), as one linear map per chunk: the interior FIR row
        and the two polynomial edge fits (mode='interp'), taken from SciPy itself applied to the
        identity so that the coefficients are the reference's."""
        from scipy.signal import savgol_filter
        if self.seamless:
            raise ValueError('--smooth-output is per-chunk Savitzky-Golay by definition: not available in '
                             'seamless mode')
        if self.plan.demod == 'iq':
            raise ValueError('--smooth-output is not available with iq output')
        w = int(window)
        if w > self.M:
            raise ValueError(f'smoothing window {w} longer than a chunk\'s {self.M} outputs')
        # SciPy applied to the identity of a longer signal gives the three linear maps it uses:
        # head rows (fit of the first w samples), the interior FIR and where its window sits
        # relative to the output (even windows are not centred), tail rows
        L = 4 * w
        S = savgol_filter(np.eye(L), w, polyorder, axis=0)
        nhead = ntail = w // 2
        k0 = 2 * w
        nz = np.nonzero(S[k0])[0]
        lo = int(nz[0]) - k0
        assert nz[-1] - nz[0] + 1 <= w and np.allclose(S[k0 + 1, k0 + 1 + lo:k0 + 1 + lo + w], S[k0, k0 + lo:k0 + lo + w])
        tab = np.concatenate([S[:nhead, :w], S[k0:k0 + 1, k0 + lo:k0 + lo + w], S[L - ntail:, L - w:]], axis=0)
        tab = np.ascontiguousarray(tab, dtype=np.float64)
        self._keep.append(tab)
        nat.check(nat.lib().sdrb_set_smooth(self._h, w, nhead, ntail, lo, tab.ctypes.data), self._h)

    def iq_gain(self, raw) -> None:
        """Advance the IQ-corrector state over whole raw chunks without producing output."""
        buf = np.frombuffer(raw, dtype=np.uint8) if not isinstance(raw, np.ndarray) else raw
        buf = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
        n = self._nchunks(buf.size)
        if n:
            nat.check(nat.lib().sdrb_iq_gain(self._h, buf.ctypes.data, n), self._h)

    def submit(self, slot: int, raw_ptr: int, nchunks: int, out_ptr: int) -> None:
        nat.check(nat.lib().sdrb_submit(self._h, slot, raw_ptr, nchunks, out_ptr), self._h)

    def wait(self, slot: int) -> None:
        nat.check(nat.lib().sdrb_wait(self._h, slot), self._h)

    def process_device(self, raw_ptr: int, nchunks: int, out_ptr: int, stream: int = 0) -> None:
        """Device pointers in/out; only enqueues work on ``stream``."""
        nat.check(nat.lib().sdrb_process_device(self._h, raw_ptr, nchunks, out_ptr, stream), self._h)

    def process_device_phases(self, raw_ptr: int, nchunks: int, out_ptr: int, phases: int,
                              stream: int = 0) -> None:
        nat.check(nat.lib().sdrb_process_device_phases(self._h, raw_ptr, nchunks, out_ptr, stream,
                                                       phases), self._h)

    def iq_export_device(self, dst_ptr: int, nsamples: int, stream: int = 0) -> None:
        """(gain.re, gain.im, nsamples) of the pass just run from a zero offset -> 3 device doubles."""
        nat.check(nat.lib().sdrb_iq_export_device(self._h, dst_ptr, float(nsamples), stream), self._h)

    def iq_prefix_device(self, gains_ptr: int, rank: int, stream: int = 0) -> None:
        """Fold the all-gathered [world][3] gains of the ranks before ``rank`` into the IQ state."""
        nat.check(nat.lib().sdrb_iq_prefix_device(self._h, gains_ptr, rank, stream), self._h)

    def reserve_sms(self, nsm: int) -> None:
        """Leave ``nsm`` SMs to a collective that runs beside the persistent kernels."""
        nat.check(nat.lib().sdrb_reserve_sms(self._h, int(nsm)), self._h)

    def set_profiling(self, on: bool) -> None:
        nat.check(nat.lib().sdrb_set_profiling(self._h, int(on)), self._h)

    def kernel_times(self) -> list[float]:
        ms = (C.c_float * 4)()
        nat.check(nat.lib().sdrb_kernel_times(self._h, ms), self._h)
        return [float(v) for v in ms]

    def decimated(self, nchunks: int) -> np.ndarray:
        """Complex decimator output of the last batch: (nchunks, R, M)."""
        y = np.empty((nchunks, self.R, self.M), dtype=np.complex128)
        nat.check(nat.lib().sdrb_read_decimated(self._h, nchunks, y.ctypes.data), self._h)
        return y

    def block_first_samples(self, nchunks: int) -> np.ndarray:
        """First raw sample of every block of the last batch as the tensor-core front end decoded it
        (exact): (nchunks, R, N // q) complex."""
        x0 = np.empty((nchunks, self.R, self.plan.Mf), dtype=np.complex128)
        nat.check(nat.lib().sdrb_read_x0(self._h, nchunks, x0.ctypes.data), self._h)
        return x0

    @property
    def iq_state(self) -> complex:
        v = (C.c_double * 2)()
        nat.check(nat.lib().sdrb_get_iq_state(self._h, v), self._h)
        return complex(v[0], v[1])

    @iq_state.setter
    def iq_state(self, off: complex) -> None:
        v = (C.c_double * 2)(off.real, off.imag)
        nat.check(nat.lib().sdrb_set_iq_state(self._h, v), self._h)

    @property
    def launches(self) -> int:
        return int(nat.lib().sdrb_launch_count(self._h))
