"""numpy emulation of the CUDA kernels' arithmetic, driven by the same ``Plan`` tables
(sdrterm_b200/plan.py).  TEST INFRASTRUCTURE: it lets the CPU suite validate the block-modal
algorithm and every table against the oracle without a GPU.  Structure mirrors the kernels:

  emu_main    <-> k_main   (per chunk x tile [x row]: decode, NCO, even/odd block sums of the
                            UNcorrected samples, IQ-EMA block aggregates, tile-local scans, partial
                            outputs + tile aggregates; the IQ corrector enters only through the
                            decoupled terms of DESIGN.md 3.3)
  emu_fixup   <-> k_fixup  (head / end segments, cross-tile carries, boundary term -> decimated y)
  emu_demod   <-> k_demod  (fm pair-phase + 2x FFT interpolation | am | re | im, output SOS)
"""
import numpy as np

from sdrterm_b200.plan import TILE_BLOCKS, Plan

_BASE = {'b': 'i1', 'B': 'u1', 'h': 'i2', 'H': 'u2', 'i': 'i4', 'I': 'u4', 'f': 'f4', 'd': 'f8'}


def decode(pl: Plan, raw: np.ndarray) -> np.ndarray:
    dt = np.dtype(_BASE[pl.enc])
    if dt.itemsize > 1:
        dt = dt.newbyteorder('>' if (pl.swap == np.little_endian) else '<')
    v = np.frombuffer(raw, dtype=dt).astype(np.float64)
    z = v[0::2] + 1j * v[1::2]
    if pl.norm is not None:
        xmin, k = pl.norm
        z = (((1.6 * (z.real - xmin)) * k) - 0.8) + 1j * ((1.6 * z.imag) * k)
    return z


def sos_segments(pl: Plan, z: np.ndarray) -> np.ndarray:
    """Output low-pass as k_demod evaluates it: 32 segments run the DF2T recurrence from a zero
    state, the segment-end states are chained with A^Lseg, and each sample then receives the
    zero-input response c A^i s_in of its segment's true initial state."""
    sos, Ls = pl.out_sos, pl.sos_Lseg
    R, M = z.shape
    ns = 2 * sos.shape[0]
    out = np.empty_like(z)
    nseg = -(-M // Ls)
    sloc = np.zeros((nseg, R, ns))
    for g in range(nseg):
        lo, hi = g * Ls, min(M, (g + 1) * Ls)
        st = np.zeros((R, ns))
        for i in range(lo, hi):
            xc = z[:, i]
            for s in range(sos.shape[0]):
                b0, b1, b2, _, a1, a2 = sos[s]
                xn = b0 * xc + st[:, 2 * s]
                st[:, 2 * s] = (b1 * xc - a1 * xn) + st[:, 2 * s + 1]
                st[:, 2 * s + 1] = b2 * xc - a2 * xn
                xc = xn
            out[:, i] = xc
        if hi - lo == Ls:
            sloc[g] = st
        else:   # short last segment: its end state is never used
            sloc[g] = st
    sin = np.zeros((R, ns))
    for g in range(nseg):
        lo, hi = g * Ls, min(M, (g + 1) * Ls)
        out[:, lo:hi] += sin @ pl.sos_CA[:hi - lo].T
        sin = sin @ pl.sos_AL.T + sloc[g]
    return out


def block_ema(pl: Plan, zb: np.ndarray) -> np.ndarray:
    """E_k = sum_j lam^(q-1-j) z_j per block: L*E_k is the offset a block adds from a zero state."""
    acc = np.zeros(zb.shape[0], dtype=np.complex128)
    for j in range(zb.shape[1]):
        acc = pl.lam * acc + zb[:, j]
    return acc


def tile_offsets(pl: Plan, blk_agg: np.ndarray):
    """Tile-local block offsets (zero at every tile start) and the tile aggregates."""
    Mf, nt = pl.Mf, pl.ntiles
    off_loc = np.zeros(Mf, dtype=np.complex128)
    tile_agg = np.zeros(nt, dtype=np.complex128)
    for t in range(nt):
        k0 = t * TILE_BLOCKS
        cnt = min(TILE_BLOCKS, Mf - k0)
        o = 0j
        for l in range(cnt):
            off_loc[k0 + l] = o
            o = pl.lam_q * o + blk_agg[k0 + l]
        tile_agg[t] = o
    return off_loc, tile_agg


def emu_main(pl: Plan, z: np.ndarray):
    """z: decoded chunk (N,).  Returns dict of per-chunk arrays written by the main kernel."""
    q, Mf, nt = pl.q, pl.Mf, pl.ntiles
    m = pl.modes
    zb = z[:q * Mf].reshape(Mf, q)
    blk_agg = pl.Liq * block_ema(pl, zb)       # offset gained over one block from zero
    off_loc, tile_agg = tile_offsets(pl, blk_agg)
    ypart = np.zeros((pl.R, Mf), dtype=np.complex128)
    Wout = np.zeros((pl.R, nt, 8), dtype=np.complex128)
    Tin = np.zeros((pl.R, nt, 8), dtype=np.complex128)
    H = q // 2
    for r in range(pl.R):
        u = zb * pl.T2[r][None, :]               # NCO only: the samples are NOT IQ-corrected here
        a = u[:, :H] + u[:, ::-1][:, :H]
        d = u[:, :H] - u[:, ::-1][:, :H]
        if q & 1:
            a = np.concatenate([a, u[:, H:H + 1]], axis=1)
            d = np.concatenate([d, np.zeros((Mf, 1))], axis=1)
        F = np.empty((Mf, 8), dtype=np.complex128)
        G = np.empty((Mf, 8), dtype=np.complex128)
        for mm in range(4):
            Er, Ei = pl.Ec[mm].real, pl.Ec[mm].imag
            Or, Oi = pl.Oc[mm].real, pl.Oc[mm].imag
            # four real sums per mode and per part, exactly what the kernel accumulates
            s1, s2, s3, s4 = a.real @ Er, a.real @ Ei, a.imag @ Er, a.imag @ Ei
            d1, d2, d3, d4 = d.real @ Or, d.real @ Oi, d.imag @ Or, d.imag @ Oi
            S_up = (s1 - s4) + 1j * (s3 + s2)
            S_lo = (s1 + s4) + 1j * (s3 - s2)
            D_up = (d1 - d4) + 1j * (d3 + d2)
            D_lo = (d1 + d4) + 1j * (d3 - d2)
            F[:, mm], G[:, mm] = S_up + D_up, S_up - D_up
            F[:, mm + 4], G[:, mm + 4] = S_lo + D_lo, S_lo - D_lo
        rb, rbT = m.rho * pl.beta[r], m.rho_p * pl.betaT[r]
        x0 = zb[:, 0]                            # first raw sample of each block (T2[0] == 1)
        for t in range(nt):
            k0 = t * TILE_BLOCKS
            cnt = min(TILE_BLOCKS, Mf - k0)
            rot = pl.T3[r][:cnt]
            Fl = F[k0:k0 + cnt] * rot[:, None]
            Gl = G[k0:k0 + cnt] * rot[:, None]
            W = np.zeros((cnt + 1, 8), dtype=np.complex128)
            for l in range(cnt):
                W[l + 1] = pl.P * W[l] + Fl[l]
            T = np.zeros((cnt + 1, 8), dtype=np.complex128)
            for l in range(cnt - 1, -1, -1):
                T[l] = pl.P * T[l + 1] + Gl[l]
            ypart[r, k0:k0 + cnt] = (W[:cnt] @ rb + T[:cnt] @ rbT
                                      + (m.g0 * x0[k0:k0 + cnt] - pl.gamma[r] * off_loc[k0:k0 + cnt]) * rot)
            Wout[r, t] = W[cnt]
            Tin[r, t] = T[0]
    return dict(ypart=ypart, Wout=Wout, Tin=Tin, tile_agg=tile_agg)


def emu_fixup(pl: Plan, z: np.ndarray, mo: dict, off_chunk: complex):
    """One chunk, all rows: (R, M) decimated complex + offset after the chunk."""
    q, Mf, nt, edge, N = pl.q, pl.Mf, pl.ntiles, pl.edge, pl.N
    m = pl.modes
    p, P = m.p, pl.P
    # offsets at tile starts
    off_tile = np.zeros(nt + 1, dtype=np.complex128)
    off_tile[0] = off_chunk
    for t in range(nt):
        kind = 1 if t == nt - 1 else 0
        cnt = pl.cnt_last if kind else TILE_BLOCKS
        off_tile[t + 1] = pl.lam_tile[kind] * off_tile[t] + mo['tile_agg'][t] if Mf else off_chunk
        _ = cnt
    # corrected head samples 0..edge (reference recurrence from the chunk-start offset)
    o = off_chunk
    xh = np.empty(edge + 1, dtype=np.complex128)
    for n in range(edge + 1):
        xh[n] = z[n] - o
        o = o + xh[n] * pl.Liq
    # corrected end-window samples ws..N-1: inside full blocks BACKWARD from the offset at q*Mf
    # (off[n] = (off[n+1] - L z[n]) / lam), in the partial block forward from it
    xe = np.empty(pl.nend, dtype=np.complex128)
    o = off_tile[nt]
    for n in range(q * Mf - 1, pl.ws - 1, -1):
        o = (o - pl.Liq * z[n]) * pl.lam_inv
        xe[n - pl.ws] = z[n] - o
    o = off_tile[nt]                       # offset at sample q*Mf
    for n in range(q * Mf, N):
        xe[n - pl.ws] = z[n] - o
        o = o + xe[n - pl.ws] * pl.Liq
    off_after = o
    if pl.rem == 0:
        off_after = off_tile[nt]
    y = np.zeros((pl.R, pl.M), dtype=np.complex128)
    for r in range(pl.R):
        xs_h = xh * pl.Ehead[r]
        xs_e = xe * pl.Eend[r]
        # head: odd extension, zi, edge samples
        ext = 2 * xs_h[0] - xs_h[edge:0:-1]
        w = m.zhat * ext[0]
        for j in range(edge):
            w = p * w + ext[j]
        # forward across tiles, in the frame of the uncorrected samples: W~ = (w + alpha s) / beta
        # with s = off e^{jwn} (n = 0: the chunk-start offset itself)
        Win = np.zeros((nt + 1, 8), dtype=np.complex128)
        Win[0] = (w + pl.alpha[r] * off_chunk) / pl.beta[r]
        s = -off_tile[:nt]
        for t in range(nt):
            kind = 1 if t == nt - 1 else 0
            cnt = pl.cnt_last if kind else TILE_BLOCKS
            Win[t + 1] = pl.Ppow[cnt] * Win[t] + pl.T1[r, t] * mo['Wout'][r, t]
        sE = off_tile[nt] * pl.phE[r]              # rotated offset at sample q*Mf
        w_end = pl.beta[r] * Win[nt] - pl.alpha[r] * sE
        # end segment: partial block (rem samples) + tail extension
        xN1 = xs_e[-1]
        tail = 2 * xN1 - xs_e[-2:-(edge + 2):-1]
        part = xs_e[pl.nend - pl.rem:] if pl.rem else xs_e[:0]
        seq = np.concatenate([part, tail])
        w = w_end.copy()
        wL1 = None
        for i, v in enumerate(seq):
            if i == len(seq) - 1:
                wL1 = w.copy()
            w = p * w + v
        wL = w
        yfL1 = np.sum(m.c * wL1) + m.d * seq[-1]
        zeta = m.zhat * yfL1 - m.xi @ wL
        T = np.zeros(8, dtype=np.complex128)
        for v in seq[::-1]:
            T = p * T + v
        Tend = T                                   # anticausal state at n = edge + q*Mf
        if pl.rem:
            k = Mf
            y[r, k] = (np.sum(m.rho * w_end) + np.sum(m.rho_p * Tend) + m.g0 * part[0]
                       + np.sum(pl.bnd[k] * zeta))
        # backward across tiles
        Tn = np.zeros((nt + 1, 8), dtype=np.complex128)
        Tn[nt] = (Tend + pl.alphaT[r] * sE) / pl.betaT[r]
        for t in range(nt - 1, -1, -1):
            kind = 1 if t == nt - 1 else 0
            cnt = pl.cnt_last if kind else TILE_BLOCKS
            Tn[t] = pl.Ppow[cnt] * Tn[t + 1] + pl.T1[r, t] * mo['Tin'][r, t]
        Wc, Tc = pl.beta[r][None, :] * Win, pl.betaT[r][None, :] * Tn      # carries as the kernels keep them
        for t in range(nt):
            kind = 1 if t == nt - 1 else 0
            cnt = pl.cnt_last if kind else TILE_BLOCKS
            k0 = t * TILE_BLOCKS
            for l in range(cnt):
                k = k0 + l
                v = pl.T1[r, t] * (mo['ypart'][r, k] + s[t] * pl.psiY[kind, r, l])
                v += np.sum(m.rho * pl.Ppow[l] * Wc[t])
                v += np.sum(m.rho_p * pl.Ppow[cnt - l] * Tc[t + 1])
                if k >= pl.k_bnd:
                    v += np.sum(pl.bnd[k] * zeta)
                y[r, k] = v
    return y, off_after


def emu_demod(pl: Plan, y: np.ndarray) -> np.ndarray:
    """(R, M) complex -> (R, M) float64, as k_demod does it."""
    M = y.shape[1]
    if pl.demod == 'fm':
        h = M >> 1
        pr = y[:, 0:2 * h:2] * np.conj(y[:, 1:2 * h:2])
        r = np.arctan2(pr.imag, pr.real)
        z = np.empty((y.shape[0], M))
        # 2x trigonometric interpolation: rfft -> halve the unpaired bin -> irfft(n=M) * 2
        X = np.fft.rfft(r, axis=1)
        m2 = h // 2 + 1
        X = X[:, :m2].copy()
        if h % 2 == 0 and M != h:
            X[:, h // 2] *= 0.5
        z[:] = np.fft.irfft(X / (h / M), n=M, axis=1)
    elif pl.demod == 'am':
        sq = y * y
        z = np.hypot(sq.real, sq.imag)
    elif pl.demod == 're':
        z = y.real.copy()
    else:
        z = y.imag.copy()
    if pl.out_sos is not None:
        zseg = sos_segments(pl, z)
        for s in range(pl.out_sos.shape[0]):
            b0, b1, b2, _, a1, a2 = pl.out_sos[s]
            z0 = np.zeros(z.shape[0])
            z1 = np.zeros(z.shape[0])
            for i in range(M):
                xc = z[:, i]
                xn = b0 * xc + z0
                z0 = (b1 * xc - a1 * xn) + z1
                z1 = b2 * xc - a2 * xn
                z[:, i] = xn
        assert np.max(np.abs(zseg - z)) <= 1e-12 * max(1e-300, np.max(np.abs(z)))
        z = zseg
    return z


def emu_stream(pl: Plan, stream: bytes, off0: complex = 0j, stale_tail: bool = True):
    """Whole byte stream -> ((R, nchunks*M) float64, (nchunks, R, M) decimated complex)."""
    raw = np.frombuffer(stream, dtype=np.uint8)
    cb = pl.chunk_bytes
    buf = np.zeros(cb, dtype=np.uint8)
    outs, ys = [], []
    off = off0
    for o in range(0, raw.size, cb):
        part = raw[o:o + cb]
        buf[:part.size] = part
        if not stale_tail and part.size < cb:
            buf[part.size:] = 0
        z = decode(pl, buf)
        mo = emu_main(pl, z)
        y, off = emu_fixup(pl, z, mo, off)
        ys.append(y)
        outs.append(emu_demod(pl, y))
    return np.concatenate(outs, axis=1), np.stack(ys), off


# ------------------------------------------------------------------------------------------------
# Tensor-core front end (k_tc): numpy twin.  The int8 GEMM is evaluated exactly in int64.
def tc_block_values(pl: Plan, tc, raw: np.ndarray, r: int = 0) -> np.ndarray:
    """raw chunk bytes -> (Mf/SB, nout + 4) float64: the linear functionals of every super-block of
    row r as k_tc's epilogue reassembles them from the int32 digit columns (the last 4: x0)."""
    nsb, K, ncol, nout = pl.Mf // tc.SB, tc.K, tc.NCOL, tc.nout
    by = np.frombuffer(raw, dtype=np.uint8)[:nsb * K].reshape(nsb, K)
    fixed = by ^ np.tile(tc.xor_mask, K // 16)[None, :]           # the sign fix-up warps
    sby = (fixed.view(np.int8) if tc.a_signed else fixed).astype(np.int64)   # the GEMM's view of the bytes
    acc = sby @ tc.Bq[r].T.astype(np.int64)                     # exact column sums
    assert np.max(np.abs(acc)) <= tc.col_l1 * (128 if tc.a_signed else 255) < 2 ** 31
    val = np.zeros((nsb, nout + 4))
    for o in range(nout):
        scale = 2.0 ** -(tc.S_yl if o >= 36 else tc.S)
        c = acc[:, ncol * o:ncol * (o + 1)]
        mid = c[:, 1] * 256 + c[:, 2]
        lo = c[:, 3] * 256 + c[:, 4]
        assert np.max(np.abs(mid)) < 2 ** 31 and np.max(np.abs(lo)) < 2 ** 31      # int32 on the device
        hi = c[:, 0] * 65536 + mid
        assert np.max(np.abs(hi)) < 2 ** 51
        # scale is a power of two: both products are exact, the sums round (device: two FMAs)
        val[:, o] = hi.astype(np.float64) * (2.0 ** 16 * scale) + (lo.astype(np.float64) * scale + tc.cst[r, o])
    x0c = 5 * nout
    for x in range(4):
        v = np.zeros(nsb, dtype=np.int64)
        for t in range(tc.isz):
            v = v * 256 + acc[:, x0c + x * tc.isz + t]
        val[:, nout + x] = v.astype(np.float64) + tc.cst[r, nout + x]
    return val


def emu_main_tc(pl: Plan, tc, raw: np.ndarray, z: np.ndarray):
    """Same outputs as emu_main, computed the way k_tc does: GEMM rows are super-blocks of two
    blocks; per tile (16 super-blocks) the exclusive scan states A (forward) and B (backward) in
    the frame of each super-block, the two block outputs from the local functionals yl_a / yl_b
    plus the scan states, the tile aggregates."""
    from sdrterm_b200 import plan as P_
    q, Mf, nt = pl.q, pl.Mf, pl.ntiles
    zb = z[:q * Mf].reshape(Mf, q)
    ypart = np.zeros((pl.R, Mf), dtype=np.complex128)
    Wout = np.zeros((pl.R, nt, 8), dtype=np.complex128)
    Tin = np.zeros((pl.R, nt, 8), dtype=np.complex128)
    tile_agg = np.zeros(nt, dtype=np.complex128)
    lq, lq2 = pl.lam_q, pl.lam_q * pl.lam_q
    for r in range(pl.R):
        v = tc_block_values(pl, tc, raw, r)
        rc = tc.rowc[r]
        F = v[:, 0:16:2] + 1j * v[:, 1:16:2]
        G = v[:, 16:32:2] + 1j * v[:, 17:32:2]
        Ea, Eab = v[:, 32] + 1j * v[:, 33], v[:, 34] + 1j * v[:, 35]
        yla, ylb = v[:, 36] + 1j * v[:, 37], v[:, 38] + 1j * v[:, 39]
        assert np.array_equal(v[:, 40] + 1j * v[:, 41], zb[0::2, 0])   # x0 comes out of the GEMM exactly
        assert np.array_equal(v[:, 42] + 1j * v[:, 43], zb[1::2, 0])
        ca, cb = rc[P_.RC_CA:P_.RC_CA + 8], rc[P_.RC_CB:P_.RC_CB + 8]
        da, db = rc[P_.RC_DA:P_.RC_DA + 8], rc[P_.RC_DB:P_.RC_DB + 8]
        Pm = rc[P_.RC_POW + 9 * np.arange(8) + 1]
        Pmb = rc[P_.RC_POW + 9 * (8 + np.arange(8)) + 1]
        rot = rc[P_.RC_ROT:P_.RC_ROT + 16]
        for t in range(nt):
            s0 = t * 16
            ea = np.zeros(16, dtype=np.complex128)
            o = 0j
            for l in range(16):
                ea[l] = o
                o = lq2 * o + pl.Liq * Eab[s0 + l]
            if r == 0:
                tile_agg[t] = o
            eb = lq * ea + pl.Liq * Ea[s0:s0 + 16]
            A = np.zeros((17, 8), dtype=np.complex128)
            for l in range(16):
                A[l + 1] = Pm * A[l] + F[s0 + l]
            B = np.zeros((17, 8), dtype=np.complex128)           # B[l] = state after super-block l from above
            for l in range(15, -1, -1):
                B[l] = Pmb * B[l + 1] + G[s0 + l]
            ya = yla[s0:s0 + 16] + A[:16] @ ca + B[1:] @ cb - rc[P_.RC_GAM] * ea
            yb = ylb[s0:s0 + 16] + A[:16] @ da + B[1:] @ db - rc[P_.RC_GAMQ] * eb
            ypart[r, t * 32:t * 32 + 32:2] = rot * ya
            ypart[r, t * 32 + 1:t * 32 + 32:2] = rot * yb
            Wout[r, t] = rc[P_.RC_AGGF] * A[16]
            Tin[r, t] = B[0]
    return dict(ypart=ypart, Wout=Wout, Tin=Tin, tile_agg=tile_agg)


def emu_stream_tc(pl: Plan, tc, stream: bytes, off0: complex = 0j):
    raw = np.frombuffer(stream, dtype=np.uint8)
    cb = pl.chunk_bytes
    buf = np.zeros(cb, dtype=np.uint8)
    outs, ys = [], []
    off = off0
    for o in range(0, raw.size, cb):
        part = raw[o:o + cb]
        buf[:part.size] = part
        z = decode(pl, buf)
        mo = emu_main_tc(pl, tc, buf, z)
        y, off = emu_fixup(pl, z, mo, off)
        ys.append(y)
        outs.append(emu_demod(pl, y))
    return np.concatenate(outs, axis=1), np.stack(ys), off
