"""Seamless mode at any decimation: a numpy twin of frames and the ragged end (TEST INFRASTRUCTURE).

``FrameTwin`` mirrors the sample-fed seamless handle (``sdrb_stream_samples*``, DESIGN.md section 11):
samples are held until they fill a frame, whole frames go through ``SeamlessTwin`` unchanged, and the
end runs the ragged last frame on a plan with its own geometry whose length-dependent tables are
derived from the whole-frame plan exactly as the handle derives them (``ragged_plan``, the mirror of
``seam_ragged_plan`` in sdrb_api.cu): pole powers and in-frame NCO phases as products of table
entries (conjugated before the frame start), ``bnd'[k] = bnd[M - M' + k] / p^(q - rem')``; then
the fold of the real end onto the last whole frame (``k_seam_fold``: anticausal state
``phi B' + p^(q Mf') T~``, ``zeta p^Lp``) and the last whole frame's fm halo from the ragged frame.
"""
from dataclasses import replace

import numpy as np
from scipy import signal

import emulator as emu
from oracle import oracle as orc
from seamless_ref import SeamlessTwin, _rows_use_nco, chunk_phasor, demodulate
from sdrterm_b200.plan import TILE_BLOCKS

_ISZ = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'i': 4, 'I': 4, 'f': 4, 'd': 8}


def ragged_plan(pl, Lp: int):
    """(plan of a ragged last frame of Lp samples, p^Lp, p^(q Mf')) from the whole-frame plan."""
    q, edge, R, TB = pl.q, pl.edge, pl.R, TILE_BLOCKS
    Mf, rem = divmod(Lp, q)
    M = Mf + (1 if rem else 0)
    nt = max(1, -(-Mf // TB))
    cnt_last = Mf - (nt - 1) * TB
    ws = min(q * Mf, Lp - 1 - edge)
    nend = Lp - ws
    pk = [pl.Pk[k] for k in range(edge + 1)]          # p^k up to edge + q - 1: p^(k-edge) p^edge
    for k in range(edge + 1, edge + q):
        pk.append(pk[k - edge] * pk[edge])

    def pw(n):
        b, j = divmod(n, q)
        return pl.Pt[b // TB] * pl.Ppow[b % TB] * pk[j]

    def phase(r, n):
        b, j = divmod(abs(n), q)
        e = pl.T1[r, b // TB] * pl.T3[r, b % TB] * pl.T2[r, j]
        return np.conj(e) if n < 0 else e

    Eend = np.array([[phase(r, ws + j) for j in range(nend)] for r in range(R)])
    phE = np.array([phase(r, q * Mf) for r in range(R)])
    bnd = pl.bnd[pl.M - M:].copy()
    if rem:
        bnd = bnd / pk[q - rem]
    pp = replace(pl, N=Lp, L=Lp + 2 * edge, Mf=Mf, rem=rem, M=M, ntiles=nt, cnt_last=cnt_last, ws=ws, nend=nend,
                 Eend=Eend, phE=phE, bnd=bnd, k_bnd=max(0, pl.k_bnd - (pl.M - M)), T1=pl.T1[:, :nt].copy(),
                 Pt=pl.Pt[:nt].copy(), lam_N=pl.lam_q ** Mf * pl.lam_j[rem],
                 lam_tile=np.array([pl.lam_tile[0], pl.lam_q ** cnt_last]))
    return pp, pw(Lp), pw(q * Mf)


class _Hist:
    """Decoded samples of the ragged frame, with the stream's samples before it at n < 0."""

    def __init__(self, z, hist):
        self.z, self.hist = z, hist

    def __getitem__(self, n):
        return self.z[n] if n >= 0 else self.hist[len(self.hist) + n]


class FrameTwin(SeamlessTwin):
    """Host mirror of a sample-fed seamless handle (fm / am / re / im): ``stream_samples(raw)`` /
    ``end()`` return (R, n) float64."""

    def __init__(self, pl, tc=None):
        super().__init__(pl, tc)
        self.pend = b''
        self.hist = np.zeros(pl.edge + 1, dtype=np.complex128)

    def stream_samples(self, raw) -> np.ndarray:
        pl, cb = self.pl, self.pl.chunk_bytes
        self.pend += bytes(raw)
        nf = len(self.pend) // cb
        if not nf:
            return np.zeros((pl.R, 0))
        whole, self.pend = self.pend[:nf * cb], self.pend[nf * cb:]
        sb = cb // pl.N
        self.hist = emu.decode(pl, np.frombuffer(whole[-(pl.edge + 1) * sb:], dtype=np.uint8))
        return self.stream(whole)

    def end(self) -> np.ndarray:
        pl = self.pl
        Lp = len(self.pend) // (pl.chunk_bytes // pl.N)
        L = self.seen * pl.N + Lp
        if 0 < L <= pl.edge or (pl.demod == 'fm' and 0 < L <= pl.q):
            self.__init__(pl, self.tc)
            raise ValueError(f'a stream of {L} samples is refused (pad {pl.edge}, fm needs two outputs)')
        if Lp == 0:
            return super().end()
        pp, pL, pQ = ragged_plan(pl, Lp)
        R, nt, m = pl.R, pp.ntiles, pl.modes
        z = emu.decode(pp, np.frombuffer(self.pend, dtype=np.uint8))
        if pp.Mf:
            mo = emu.emu_main(pp, z)
        else:   # a partial block only: no front end, zero tile aggregates
            mo = dict(ypart=np.zeros((R, 0), dtype=np.complex128), Wout=np.zeros((R, 1, 8), dtype=np.complex128),
                      Tin=np.zeros((R, 1, 8), dtype=np.complex128), tile_agg=np.zeros(1, dtype=np.complex128))
        offt = np.zeros(nt + 1, dtype=np.complex128)
        offt[0] = self.off
        for t in range(nt):
            offt[t + 1] = pp.lam_tile[1 if t == nt - 1 else 0] * offt[t] + mo['tile_agg'][t]
        A = np.zeros((R, 8), dtype=np.complex128)
        B = np.zeros((R, 8), dtype=np.complex128)
        for t in range(nt):
            cnt = pp.cnt_last if t == nt - 1 else TILE_BLOCKS
            A = pl.Ppow[cnt] * A + pp.T1[:, t, None] * mo['Wout'][:, t]
        for t in range(nt - 1, -1, -1):
            cnt = pp.cnt_last if t == nt - 1 else TILE_BLOCKS
            B = pl.Ppow[cnt] * B + pp.T1[:, t, None] * mo['Tin'][:, t]
        phi = chunk_phasor(pl, self.seen)
        if self.seen == 0:
            self.G = emu.emu_head(pp, z, offt[0])
            self.sos_state = np.zeros((R, 0 if pl.out_sos is None else pl.sos_AM.shape[0]))
        G = self.G
        Gend = pQ * G + phi[:, None] * A                  # forward state at q Mf' (k_seam_fscan, PN row p^(q Mf'))
        e = emu.emu_end(pp, _Hist(z, self.hist), offt[nt], np.conj(phi)[:, None] * Gend)
        Tt, zeta = phi[:, None] * e['Tt'], phi[:, None] * e['zeta']
        # the ragged frame's outputs (k_seam_carry / k_seam_y on its plan, k_seam_tail's partial block)
        yp = np.zeros((R, pp.M), dtype=np.complex128)
        s = -offt[:nt] if pl.correct_iq else np.zeros(nt)
        for r in range(R):
            ph = phi[r]
            Win = np.zeros((nt + 1, 8), dtype=np.complex128)
            Win[0] = np.conj(ph) * G[r]
            for t in range(nt):
                cnt = pp.cnt_last if t == nt - 1 else TILE_BLOCKS
                Win[t + 1] = pl.Ppow[cnt] * Win[t] + pp.T1[r, t] * mo['Wout'][r, t]
            Tn = np.zeros((nt + 1, 8), dtype=np.complex128)
            Tn[nt] = np.conj(ph) * Tt[r]
            for t in range(nt - 1, -1, -1):
                cnt = pp.cnt_last if t == nt - 1 else TILE_BLOCKS
                Tn[t] = pl.Ppow[cnt] * Tn[t + 1] + pp.T1[r, t] * mo['Tin'][r, t]
            Wc, Tc = pl.beta[r] * Win, pl.betaT[r] * Tn
            for t in range(nt if pp.Mf else 0):
                cnt = pp.cnt_last if t == nt - 1 else TILE_BLOCKS
                l = np.arange(cnt)
                k = t * TILE_BLOCKS + l
                v = pp.T1[r, t] * (mo['ypart'][r, k] + s[t] * pl.psiY[1 if t == nt - 1 else 0, r, l])
                v += (pl.Ppow[l] * Wc[t]) @ m.rho + (pl.Ppow[cnt - l] * Tc[t + 1]) @ m.rho_p
                v += pp.bnd[k] @ (np.conj(ph) * zeta[r])
                yp[r, k] = ph * v
            if pp.rem:
                yp[r, pp.Mf] = ph * (np.sum(m.rho * e['w'][r]) + np.sum(m.rho_p * e['T'][r])
                                     + np.sum(pp.bnd[pp.Mf] * e['zeta'][r]) + m.g0 * e['x0'][r])
        # the real end moved onto the last whole frame (k_seam_fold); its halo is the ragged frame's y[0]
        end = (phi[:, None] * B + pQ * Tt, pL * zeta)
        outs, ylast = [], None
        while self.win:
            y, last = self._y(0, end)
            if last:
                y[:, pl.M] = yp[:, 0]
                ylast = y[:, pl.M - 1]
            outs.append(self._demod(y, False))
            self.win.pop(0)
            self.emitted += 1
        if pl.demod == 'fm':
            d = np.empty((R, pp.M))
            if pp.M == 1:
                d[:, 0] = np.angle(ylast * np.conj(yp[:, 0]))
            else:
                d[:, :-1] = np.angle(yp[:, :-1] * np.conj(yp[:, 1:]))
                d[:, -1] = d[:, -2]
        elif pl.demod == 'am':
            d = np.abs(yp * yp)
        elif pl.demod == 're':
            d = yp.real.copy()
        else:
            d = yp.imag.copy()
        if pl.out_sos is not None:
            d = emu.sos_segments(pp, d) + self.sos_state @ pl.sos_CAM[:pp.M].T
        outs.append(d)
        self.__init__(pl, self.tc)
        return np.concatenate(outs, axis=1)


def ragged_oracle(kw: dict, body: bytes) -> np.ndarray:
    """seamless_oracle of a stream of any whole number of samples (fm / am / re / im): decode and
    correct as the reader does over whole chunks (zero-padded), keep the stream's L samples."""
    ch = orc.Chain(**kw)
    L = len(body) // (2 * _ISZ[kw['enc']])
    st = np.frombuffer(body + bytes(-len(body) % ch.chunk_bytes), dtype=np.uint8)
    z = np.concatenate([ch.ingest(st[o:o + ch.chunk_bytes]).copy() for o in range(0, st.size, ch.chunk_bytes)])[:L]
    n = np.arange(L, dtype=np.int64)
    ys = [signal.decimate(z * np.exp(-2j * np.pi * (((int(f) * n) % kw['fs']) / kw['fs'])) if on else z, kw['dec'])
          for f, on in zip(ch.rows, _rows_use_nco(kw, ch.rows))]
    return demodulate(kw, np.array(ys))
