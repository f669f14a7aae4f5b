"""Seamless streaming mode: the oracle and the numpy twin of its finish stage (TEST INFRASTRUCTURE).

``seamless_oracle`` is the contract of DESIGN.md section 11 restated from ``oracle/`` and SciPy on
the concatenated stream: decode / normalise / IQ-correct chunk by chunk exactly as the reader does
(the corrector already runs over the whole stream), the NCO with the exact global phase
``exp(-2 pi i ((f n) mod fs) / fs)``, ``scipy.signal.decimate`` over the whole stream, the
demodulator (fm: ``angle(y[k] conj(y[k+1]))``, last sample repeated), the output low-pass
``sosfilt`` over the whole stream from a zero state.

``SeamlessTwin`` mirrors the device decomposition call by call (sdrb_seamless.cuh): the chunk-local
front-end outputs of ``tests/emulator.py`` rotated by one phasor per (chunk, row), a forward scan
of the chunk aggregates, the fixed-horizon anticausal window over the next D chunks, the stream's
two real boundaries, the demodulator with its one-sample halo and the output SOS as a zero-state
response plus the response to the carried state.
"""
import numpy as np
from scipy import signal

import emulator as emu
from oracle import oracle as orc
from sdrterm_b200.plan import TILE_BLOCKS


def _rows_use_nco(kw, rows):
    return [bool(kw['simo'] or f) for f in rows]


def seamless_decimated(kw: dict, stream: bytes) -> tuple[np.ndarray, complex]:
    """(R, C*M) complex decimator output over the whole stream, and the final IQ offset."""
    ch = orc.Chain(**kw)
    st = np.frombuffer(stream, dtype=np.uint8)
    zs = [ch.ingest(st[o:o + ch.chunk_bytes]).copy() for o in range(0, st.size, ch.chunk_bytes)]
    z = np.concatenate(zs)
    n = np.arange(z.size, dtype=np.int64)
    ys = []
    for f, on in zip(ch.rows, _rows_use_nco(kw, ch.rows)):
        u = z * np.exp(-2j * np.pi * (((int(f) * n) % kw['fs']) / kw['fs'])) if on else z
        ys.append(signal.decimate(u, kw['dec']))
    return np.array(ys), complex(ch._off[0])


def discriminator(y: np.ndarray) -> np.ndarray:
    """fm of the seamless mode: d[k] = angle(y[k] conj(y[k+1])), d[K-1] = d[K-2]."""
    d = np.empty(y.shape)
    d[..., :-1] = np.angle(y[..., :-1] * np.conj(y[..., 1:]))
    d[..., -1] = d[..., -2]
    return d


def demodulate(kw: dict, y: np.ndarray) -> np.ndarray:
    if kw['demod'] == 'fm':
        d = discriminator(y)
    elif kw['demod'] == 'am':
        d = np.abs(y * y)
    elif kw['demod'] == 're':
        d = y.real.copy()
    else:
        d = y.imag.copy()
    if kw['demod'] in ('fm', 'am'):
        sos = orc.output_filter_sos(kw['fs'] // kw['dec'], kw['omega_out'])
        d = signal.sosfilt(sos, d, axis=-1)
    return d


def seamless_oracle(kw: dict, stream: bytes) -> tuple[np.ndarray, complex]:
    """(R, C*M) float64 seamless output of a whole-chunk stream, and the final IQ offset."""
    y, off = seamless_decimated(kw, stream)
    return demodulate(kw, y), off


# ------------------------------------------------------------------------------------------------
def chunk_phasor(pl, g: int) -> np.ndarray:
    """phi_{g,r} = exp(-2 pi i ((f_r N g) mod fs) / fs) per row, exact integer phase."""
    idx = (pl.chunk_step.astype(object) * g) % pl.fs
    return np.array([np.exp(-2j * np.pi * (int(v) / pl.fs)) for v in idx])


class SeamlessTwin:
    """Host mirror of the seamless handle: ``stream(raw)`` / ``end()`` return (R, k*M) float64."""

    def __init__(self, pl, tc=None):
        assert pl.seamless and pl.rem == 0
        self.pl, self.tc = pl, tc
        self.D = pl.lookahead
        self.win = []             # unemitted chunks: dict(z, mo, offt, A, B, g, phi, G)
        self.G = None             # forward state at the next new chunk (global frame), (R, 8)
        self.seen = 0
        self.emitted = 0
        self.off = 0j
        self.sos_state = None

    # -- per chunk: front end (chunk-local), IQ offsets, chunk aggregates
    def _front(self, raw: np.ndarray, g: int):
        pl = self.pl
        z = emu.decode(pl, raw)
        mo = emu.emu_main_tc(pl, self.tc, raw, z) if self.tc is not None else emu.emu_main(pl, z)
        nt = pl.ntiles
        offt = np.zeros(nt + 1, dtype=np.complex128)
        offt[0] = self.off
        for t in range(nt):
            offt[t + 1] = pl.lam_tile[1 if t == nt - 1 else 0] * offt[t] + mo['tile_agg'][t]
        self.off = offt[nt]
        A = np.zeros((pl.R, 8), dtype=np.complex128)
        B = np.zeros((pl.R, 8), dtype=np.complex128)
        for t in range(nt):
            cnt = pl.cnt_last if t == nt - 1 else TILE_BLOCKS
            A = pl.Ppow[cnt] * A + pl.T1[:, t, None] * mo['Wout'][:, t]
        for t in range(nt - 1, -1, -1):
            cnt = pl.cnt_last if t == nt - 1 else TILE_BLOCKS
            B = pl.Ppow[cnt] * B + pl.T1[:, t, None] * mo['Tin'][:, t]
        return dict(z=z, mo=mo, offt=offt, A=A, B=B, g=g, phi=chunk_phasor(pl, g))

    def _head(self, c) -> np.ndarray:
        """Forward state at sample 0 of the stream (odd extension, zi), frame of the uncorrected samples."""
        return emu.emu_head(self.pl, c['z'], c['offt'][0])

    def _tail(self, c, Gend):
        """True end of the stream: anticausal state after the last chunk and zeta (global frame)."""
        e = emu.emu_end(self.pl, c['z'], c['offt'][self.pl.ntiles], np.conj(c['phi'])[:, None] * Gend)
        return c['phi'][:, None] * e['Tt'], c['phi'][:, None] * e['zeta']

    # -- one chunk's decimated output (global frame) with its carry-ins, plus the halo sample
    def _y(self, i, end):
        pl, m = self.pl, self.pl.modes
        c = self.win[i]
        nt, D = pl.ntiles, self.D
        last = end is not None and i == len(self.win) - 1
        known = end is not None and len(self.win) - 1 - i <= D
        J = (len(self.win) - 1 - i) if known else D
        Tg = end[0].copy() if known else np.zeros((pl.R, 8), dtype=np.complex128)
        for j in range(J, 0, -1):
            nx = self.win[i + j]
            Tg = pl.PN[1] * Tg + nx['phi'][:, None] * nx['B']
        Zc = end[1] * pl.PN[len(self.win) - 1 - i] if known else None
        y = np.zeros((pl.R, pl.M + 1), dtype=np.complex128)
        s = -c['offt'][:nt] if pl.correct_iq else np.zeros(nt)
        for r in range(pl.R):
            ph = c['phi'][r]
            Win = np.zeros((nt + 1, 8), dtype=np.complex128)
            Win[0] = np.conj(ph) * c['G'][r]
            for t in range(nt):
                cnt = pl.cnt_last if t == nt - 1 else TILE_BLOCKS
                Win[t + 1] = pl.Ppow[cnt] * Win[t] + pl.T1[r, t] * c['mo']['Wout'][r, t]
            Tn = np.zeros((nt + 1, 8), dtype=np.complex128)
            Tn[nt] = np.conj(ph) * Tg[r]
            for t in range(nt - 1, -1, -1):
                cnt = pl.cnt_last if t == nt - 1 else TILE_BLOCKS
                Tn[t] = pl.Ppow[cnt] * Tn[t + 1] + pl.T1[r, t] * c['mo']['Tin'][r, t]
            Wc, Tc = pl.beta[r] * Win, pl.betaT[r] * Tn
            for t in range(nt):
                cnt = pl.cnt_last if t == nt - 1 else TILE_BLOCKS
                l = np.arange(cnt)
                k = t * TILE_BLOCKS + l
                v = pl.T1[r, t] * (c['mo']['ypart'][r, k] + s[t] * pl.psiY[1 if t == nt - 1 else 0, r, l])
                v += (pl.Ppow[l] * Wc[t]) @ m.rho + (pl.Ppow[cnt - l] * Tc[t + 1]) @ m.rho_p
                if Zc is not None:
                    v += pl.bnd[k] @ (np.conj(ph) * Zc[r])
                y[r, k] = ph * v
            if not last:
                # block 0 of the next chunk, from this chunk's horizon
                nx = self.win[i + 1]
                off1 = c['offt'][nt] if pl.correct_iq else 0j
                v = (np.sum(m.rho * pl.beta[r] * nx['G'][r]) + np.sum(m.rho_p * pl.betaT[r] * Tg[r])
                     + nx['phi'][r] * (m.g0 * nx['z'][0] - pl.gamma[r] * off1))
                if known:
                    v += pl.bnd[0] @ (end[1][r] * pl.PN[len(self.win) - 2 - i])
                y[r, pl.M] = v
        return y, last

    def _demod(self, y, last):
        pl = self.pl
        if pl.demod == 'fm':
            d = np.angle(y[:, :-1] * np.conj(y[:, 1:]))
            if last:
                d[:, -1] = d[:, -2]
        elif pl.demod == 'am':
            d = np.abs(y[:, :-1] * y[:, :-1])
        elif pl.demod == 're':
            d = y[:, :-1].real.copy()
        else:
            d = y[:, :-1].imag.copy()
        if pl.out_sos is None:
            return d
        # zero-state response of this chunk + response to the carried state; state chained by A^M
        zs = emu.sos_segments(pl, d)
        ns = pl.sos_AM.shape[0]
        e = np.zeros((pl.R, ns))
        for g in range(-(-pl.M // pl.sos_Lseg)):
            seg = np.zeros((pl.R, ns))
            st = np.zeros((pl.R, ns))
            for i_ in range(g * pl.sos_Lseg, min(pl.M, (g + 1) * pl.sos_Lseg)):
                xc = d[:, i_]
                for s_ in range(pl.out_sos.shape[0]):
                    b0, b1, b2, _, a1, a2 = pl.out_sos[s_]
                    xn = b0 * xc + st[:, 2 * s_]
                    st[:, 2 * s_] = (b1 * xc - a1 * xn) + st[:, 2 * s_ + 1]
                    st[:, 2 * s_ + 1] = b2 * xc - a2 * xn
                    xc = xn
            seg = st
            e = e @ pl.sos_AL.T + seg
        out = zs + self.sos_state @ pl.sos_CAM.T
        self.sos_state = self.sos_state @ pl.sos_AM.T + e
        return out

    def _emit(self, upto: int, end) -> np.ndarray:
        outs = []
        while self.emitted < upto:
            y, last = self._y(0, end)
            outs.append(self._demod(y, last))
            self.win.pop(0)
            self.emitted += 1
        if not outs:
            return np.zeros((self.pl.R, 0))
        return np.concatenate(outs, axis=1)

    def stream(self, raw) -> np.ndarray:
        pl = self.pl
        raw = np.frombuffer(raw, dtype=np.uint8)
        cb = pl.chunk_bytes
        assert raw.size % cb == 0
        for o in range(0, raw.size, cb):
            c = self._front(raw[o:o + cb], self.seen)
            if self.seen == 0:
                self.G = self._head(c)
                ns = 0 if pl.out_sos is None else pl.sos_AM.shape[0]
                self.sos_state = np.zeros((pl.R, ns))
            c['G'] = self.G
            self.G = pl.PN[1] * self.G + c['phi'][:, None] * c['A']
            self.win.append(c)
            self.seen += 1
        return self._emit(max(0, self.seen - self.D), None)

    def end(self) -> np.ndarray:
        if not self.win:
            out = np.zeros((self.pl.R, 0))
        else:
            end = self._tail(self.win[-1], self.G)
            out = self._emit(self.seen, end)
        self.__init__(self.pl, self.tc)
        return out
