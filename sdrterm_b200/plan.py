"""Host-side plan for the B200 decimation chain: every table the CUDA kernels consume.

The reference filters each 131072-byte chunk independently with SciPy's
``decimate(x, q)`` = zero-phase ``sosfiltfilt`` of a Chebyshev-I order-8 low-pass followed by
``[::q]`` (src/dsp/dsp_processor.py:147; SciPy _signaltools.py:5091-5203, 5206-5369).  A
sample-serial IIR is a poor fit for a GPU, and only every q-th output is kept, so the device
path evaluates the *same linear operator* in block form (DESIGN.md section 3):

* the cascade is diagonalised once, here, in 50-digit arithmetic (mpmath): poles ``p_i``,
  normalised modal output weights ``c_i``, ``kappa_i = H(1/p_i)``, ``rho_i = c_i*kappa_i``;
* forward modal states ``w_i[n+1] = p_i w_i[n] + x[n]`` and anticausal states
  ``T_i[n] = p_i T_i[n+1] + x[n]`` are advanced one *block* of q samples at a time,
  ``W <- p^q W + F``, ``T <- p^q T + G`` with ``F = sum_j p^(q-1-j) u_j``, ``G = sum_j p^j u_j``;
  both come from one pass over the block through the even/odd split
  ``F,G = S +- D``, ``S = sum_j Ec_j (u_j + u_(q-1-j))``, ``D = sum_j Oc_j (u_j - u_(q-1-j))``;
* the decimated output at a block start is
  ``y[n] = sum_i rho_i w_i[n] + sum_i (rho_i/p_i) T_i[n] + g0 x[n] + sum_i c_i p_i^(L-1-n) zeta_i``
  where the last term carries sosfiltfilt's finite-length / ``zi`` boundary condition.

Filter *design* (cheby1, sosfilt_zi, ellip) is SciPy's, exactly as in the reference, so the
coefficients are identical to the oracle's.  Nothing here touches the GPU.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

mp = None          # mpmath and scipy.signal are imported on first use (_heavy): a process that finds
_sig = None        # its plan in the cache (cached_plan) never pays for them


def _heavy():
    global mp, _sig
    if mp is None:
        import mpmath
        from scipy import signal
        mp, _sig = mpmath, signal

TILE_BLOCKS = 32          # one warp: lane <-> block
CHUNK_BYTES = 131072      # src/misc/read_file.py:38
_ITEMSIZE = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'i': 4, 'I': 4, 'f': 4, 'd': 8, 'Z': 8}


def _c(x) -> complex:
    return complex(mp.re(x), mp.im(x))


def _cascade_state_space(sos):
    """Exact (A, b, c, d) of the DF2T cascade, state = [z0_1, z1_1, z0_2, z1_2, ...] -- the
    same variables SciPy's _sosfilt carries, so sosfilt_zi maps onto it directly."""
    ns = len(sos)
    n = 2 * ns
    A = mp.zeros(n, n)
    b = mp.zeros(n, 1)
    # u (section input) as a linear form over [state..., x]
    u = [mp.mpf(0)] * n + [mp.mpf(1)]
    for k in range(ns):
        b0, b1, b2, a0, a1, a2 = [mp.mpf(float(v)) for v in sos[k]]
        assert a0 == 1
        y = [b0 * t for t in u]
        y[2 * k] += 1
        z0 = [b1 * t - a1 * s for t, s in zip(u, y)]
        z0[2 * k + 1] += 1
        z1 = [b2 * t - a2 * s for t, s in zip(u, y)]
        for j in range(n):
            A[2 * k, j] = z0[j]
            A[2 * k + 1, j] = z1[j]
        b[2 * k] = z0[n]
        b[2 * k + 1] = z1[n]
        u = y
    c = mp.matrix(1, n)
    for j in range(n):
        c[0, j] = u[j]
    return A, b, c, u[n]


@dataclass
class FilterModes:
    """Normalised modal form of the decimation low-pass (poles 0..3 upper half plane, 4..7 their
    conjugates, same order)."""
    p: np.ndarray          # (8,) complex
    c: np.ndarray          # (8,) normalised output weights c_i (input weight 1 per mode)
    kappa: np.ndarray      # (8,) H(1/p_i)
    rho: np.ndarray        # (8,) c_i * kappa_i
    rho_p: np.ndarray      # (8,) rho_i / p_i
    zhat: np.ndarray       # (8,) sosfilt_zi in normalised modal coordinates
    xi: np.ndarray         # (8,8) c_l / (1 - p_i p_l)   [i, l]
    d: float
    g0: float
    mp_p: list = field(repr=False, default=None)   # high-precision poles for table building
    mp_c: list = field(repr=False, default=None)


def filter_modes(sos: np.ndarray, zi: np.ndarray, dps: int = 50) -> FilterModes:
    _heavy()
    mp.mp.dps = dps
    A, b, c, d = _cascade_state_space(sos)
    n = A.rows
    E, ER = mp.eig(A)
    idx_up = sorted([i for i in range(n) if mp.im(E[i]) > 0], key=lambda i: -abs(mp.im(E[i])))
    if 2 * len(idx_up) != n:
        raise ValueError('decimation filter must have complex-conjugate pole pairs only')
    order = list(idx_up)
    for i in idx_up:  # conjugate partner
        j = min((j for j in range(n) if mp.im(E[j]) < 0), key=lambda j: abs(E[j] - mp.conj(E[i])))
        order.append(j)
    p = [E[i] for i in order]
    V = mp.matrix(n, n)
    for col, i in enumerate(order):
        for r in range(n):
            V[r, col] = ER[r, i]
    beta = mp.lu_solve(V, b)
    zflat = mp.matrix([mp.mpf(float(v)) for v in np.asarray(zi).reshape(-1)])
    zmod = mp.lu_solve(V, zflat)
    cV = c * V
    chat = [cV[0, i] * beta[i] for i in range(n)]
    zhat = [zmod[i] / beta[i] for i in range(n)]
    kappa = [d + p[i] * sum(chat[l] / (1 - p[i] * p[l]) for l in range(n)) for i in range(n)]
    rho = [chat[i] * kappa[i] for i in range(n)]
    chi = [(kappa[l] - d) / p[l] for l in range(n)]
    g0 = d * d + sum(chi[l] * chat[l] for l in range(n)) - sum(rho[i] / p[i] for i in range(n))
    xi = np.array([[_c(chat[l] / (1 - p[i] * p[l])) for l in range(n)] for i in range(n)])
    return FilterModes(p=np.array([_c(v) for v in p]), c=np.array([_c(v) for v in chat]),
                       kappa=np.array([_c(v) for v in kappa]), rho=np.array([_c(v) for v in rho]),
                       rho_p=np.array([_c(rho[i] / p[i]) for i in range(n)]),
                       zhat=np.array([_c(v) for v in zhat]), xi=xi, d=float(d),
                       g0=float(mp.re(g0)), mp_p=p, mp_c=chat)


def _phasor(w: float, n) -> np.ndarray:
    """exp(1j*w*n) with the product formed in 80-bit arithmetic (w is the reference's rounded
    double; the reference itself rounds w*n to double before exp, so it deviates from these
    values by <= ulp(w*n)/2 in phase -- DESIGN.md section 5)."""
    ph = np.longdouble(w) * np.asarray(n, dtype=np.longdouble)
    return (np.cos(ph) + 1j * np.sin(ph)).astype(np.complex128)


def _phasor_vec(w: np.ndarray, n: int) -> np.ndarray:
    """exp(1j*w[r]*n) per row (same 80-bit product as _phasor)."""
    return np.array([_phasor(wr, n) for wr in w]).reshape(-1)


@dataclass
class Plan:
    # geometry
    enc: str
    swap: bool
    fs: int
    q: int
    N: int
    edge: int
    L: int
    Mf: int            # full blocks
    rem: int           # samples in the trailing partial block
    M: int             # outputs per chunk-row = ceil(N/q)
    ntiles: int
    cnt_last: int      # blocks in the last tile
    Hq: int            # pairs per block = ceil(q/2)
    rows_hz: list
    R: int
    # filter
    sos: np.ndarray
    zi: np.ndarray
    modes: FilterModes
    P: np.ndarray          # (8,) p^q
    Ec: np.ndarray         # (4, Hq) complex: even-part coefficients, upper poles
    Oc: np.ndarray         # (4, Hq) complex: odd-part coefficients
    Ppow: np.ndarray       # (TILE_BLOCKS+1, 8) P^l
    Pk: np.ndarray         # (max(edge+1, edge+rem), 8) p^k
    Pt: np.ndarray         # (ntiles, 8) p^(q*TILE_BLOCKS*m)
    bx: np.ndarray         # (8,) p^edge / kappa
    bnd: np.ndarray        # (M, 8) c_i p_i^(L-1-n_k)
    k_bnd: int             # first k whose boundary term is not negligible
    # IQ corrector
    correct_iq: bool
    Liq: float
    lam: float
    lam_j: np.ndarray      # (q+1,) lam^j
    lam_q: float
    lam_N: float
    lam_inv: float         # 1/lam (backward EMA over the descending half of a block)
    lam_k: np.ndarray      # (33,) lam^k
    mu_k: np.ndarray       # (33,) lam^-k
    RL: int                # pairs per DMMA k-lane = ceil(Hq/4): lane k owns pairs [k*RL, (k+1)*RL)
    run_len: np.ndarray    # (8,) samples per run, in sample order (4 ascending + 4 descending runs)
    lam_run: np.ndarray    # (8,) lam^run_len
    # normalisation (read_file.py:82-96), None when off
    norm: tuple | None
    # per row
    w: np.ndarray          # (R,) phase increment per sample (reference's rounded double)
    use_nco: np.ndarray    # (R,) bool: False reproduces "no shift when centre == 0"
    T2: np.ndarray         # (R, q)
    T3: np.ndarray         # (R, TILE_BLOCKS+1)
    T1: np.ndarray         # (R, ntiles)
    Ehead: np.ndarray      # (R, edge+1)  phases of samples 0..edge
    Eend: np.ndarray       # (R, nend)    phases of samples ws..N-1
    ws: int
    nend: int
    # IQ corrector decoupled from the modal sums (DESIGN.md 3.3): with s[n] = off[n] e^{jwn} and
    # mu = lam e^{jw}, the corrected modal states are w_i = beta_i W~_i - alpha_i s,
    # T_i = betaT_i T~_i - alphaT_i s with W~, T~ driven by the UNcorrected rotated samples, and
    # y = sum rho_i beta_i W~_i + sum rho'_i betaT_i T~_i + g0 u~ - gamma s
    alpha: np.ndarray      # (R, 8)  1 / (mu - p_i)
    beta: np.ndarray       # (R, 8)  1 + alpha_i L e^{jw}
    alphaT: np.ndarray     # (R, 8)  1 / (1 - p_i mu)
    betaT: np.ndarray      # (R, 8)  1 - p_i alphaT_i L e^{jw}
    gamma: np.ndarray      # (R,)    sum rho_i alpha_i + sum rho'_i alphaT_i + g0  (0 when IQ correction is off)
    phE: np.ndarray        # (R,)    e^{j w q Mf}: NCO phase at the end of the full blocks
    psiY: np.ndarray       # (2, R, TILE_BLOCKS)  gamma mu^(q l): tile-start offset -> block l's output
    lam_tile: np.ndarray   # (2,) lam^(q*cnt)
    # demod / output
    demod: str
    out_sos: np.ndarray | None
    big_endian_out: bool
    fm_interp: np.ndarray | None = None   # (M, M>>1) dense resample matrix, non-power-of-two FM only
    sos_Lseg: int = 0                     # output SOS evaluated in 32 segments of this length
    sos_AL: np.ndarray | None = None      # (ns, ns) A^Lseg of the output cascade (ns = 2*sections)
    sos_CA: np.ndarray | None = None      # (Lseg, ns) c A^i
    sos_AP: np.ndarray | None = None      # (5, ns, ns) (A^Lseg)^(2^lv)
    # seamless streaming (DESIGN.md section 11): the whole stream is filtered, not each chunk
    seamless: bool = False
    lookahead: int = 0                    # D: chunk c is final once chunks c+1 .. c+D exist
    chunk_step: np.ndarray | None = None  # (R,) int64: (f_r * N) mod fs, NCO phase step per chunk
    PN: np.ndarray | None = None          # (D+1, 8) p_i^(N j): a modal state moved j whole chunks
    sos_AM: np.ndarray | None = None      # (ns, ns) A^M of the output cascade: its state moved one chunk
    sos_CAM: np.ndarray | None = None     # (M, ns) c A^i, i < M
    # single sideband (usb / lsb; DESIGN.md section 12): out_sos is the prototype, the band-pass is
    # h[m] e^{j Omega m}; the kernels run it in the Weaver frame and need only e^{j Omega k}
    ssb_omega: float = 0.0                # Omega = +pi B / fs_d (usb), -pi B / fs_d (lsb)
    ssb_rot: np.ndarray | None = None     # (M+1,) e^{j Omega k}, k = 0..M

    @property
    def chunk_bytes(self) -> int:
        return self.N * 2 * _ITEMSIZE[self.enc]

    @property
    def W(self) -> int:
        """Doubles per chunk and row of the output: 2M for iq ((Re, Im) interleaved), M otherwise."""
        return 2 * self.M if self.demod == 'iq' else self.M


def reference_w(f_hz: int, fs: int) -> float:
    """Phase increment per sample exactly as the reference forms it:
    ``-2j * pi * (f / fs)`` (dsp_processor.py:187, vfo_processor.py:48)."""
    return float((-2j * np.pi * (f_hz / fs)).imag)


def ssb_omega(demod: str, omega_out: int, fs_d: int) -> float:
    """The single-sideband rotation Omega = +pi B / fs_d (usb) or -pi B / fs_d (lsb), B = omegaOut."""
    om = np.pi * omega_out / fs_d
    return float(om if demod == 'usb' else -om)


LOOKAHEAD_TOL = 1e-13     # truncated anticausal tail of the seamless mode, relative to the input scale


def lookahead_bound(p, rho_p, N: int, D: int) -> float:
    """sum_i |rho_i/p_i| |p_i|^(D N) / (1 - |p_i|): what the anticausal modes of the samples after
    chunk c+D can still add to an output of chunk c, per unit of input magnitude."""
    a = np.abs(np.asarray(p))
    return float(np.sum(np.abs(np.asarray(rho_p)) * a ** (D * N) / (1 - a)))


def lookahead_chunks(p, rho_p, N: int, tol: float = LOOKAHEAD_TOL) -> int:
    """Smallest D >= 1 whose truncation bound is <= tol."""
    D = 1
    while lookahead_bound(p, rho_p, N, D) > tol:
        D += 1
    return D


def seamless_frame_samples(N: int, q: int) -> int:
    """Samples per frame of the seamless mode for chunks of N samples at decimation q: the most
    whole tiles (32 blocks of q samples) that fit a chunk, 32 q floor(N / (32 q)).  Equal to N for
    every power-of-two q that divides N/32.  The seamless pipeline runs on frames, not on the reader's
    chunks, so any q works (DESIGN.md section 11)."""
    return TILE_BLOCKS * q * (N // (TILE_BLOCKS * q))


def build_plan(fs: int, enc: str, dec: int, rows_hz, *, simo: bool = False, swap: bool = False,
               correct_iq: bool = False, normalize: bool = False, impedance: int = 50,
               demod: str = 'fm', omega_out: int = 12500, chunk_bytes: int = CHUNK_BYTES,
               big_endian_out: bool | None = None, seamless: bool = False) -> Plan:
    _heavy()
    if dec < 2:
        raise ValueError('Decimation must be at least 2.')
    if enc not in _ITEMSIZE:
        raise ValueError(f'unknown encoding {enc!r}')
    q = int(dec)
    N = chunk_bytes // (2 * _ITEMSIZE[enc])
    if seamless and N % q:
        raise ValueError(f'seamless mode needs the decimation to divide the {N} samples of a chunk '
                         f'(-d {q} leaves a ragged block); use a power of two')
    sos = np.ascontiguousarray(_sig.cheby1(8, 0.05, 0.8 / q, output='sos'), dtype=np.float64)
    zi = np.ascontiguousarray(_sig.sosfilt_zi(sos), dtype=np.float64)
    nsec = sos.shape[0]
    edge = 3 * (2 * nsec + 1 - min(int((sos[:, 2] == 0).sum()), int((sos[:, 5] == 0).sum())))
    if N <= edge + 1:
        raise ValueError(f'chunk of {N} samples is not longer than the filter pad ({edge})')
    L = N + 2 * edge
    Mf, rem = divmod(N, q)
    M = Mf + (1 if rem else 0)
    ntiles = max(1, -(-Mf // TILE_BLOCKS))
    cnt_last = Mf - (ntiles - 1) * TILE_BLOCKS
    Hq = (q + 1) // 2

    modes = filter_modes(sos, zi)
    pm = modes.mp_p
    n8 = len(pm)
    nu = n8 // 2
    P = np.array([_c(pm[i] ** q) for i in range(n8)])
    Ec = np.zeros((nu, Hq), dtype=np.complex128)
    Oc = np.zeros((nu, Hq), dtype=np.complex128)
    for m in range(nu):
        for j in range(Hq):
            if 2 * j == q - 1:          # middle sample of an odd block
                Ec[m, j] = _c(pm[m] ** j)
            else:
                Ec[m, j] = _c((pm[m] ** (q - 1 - j) + pm[m] ** j) / 2)
                Oc[m, j] = _c((pm[m] ** (q - 1 - j) - pm[m] ** j) / 2)
    Ppow = np.array([[_c(pm[i] ** (q * l)) for i in range(n8)] for l in range(TILE_BLOCKS + 1)])
    Pk = np.array([[_c(pm[i] ** k) for i in range(n8)] for k in range(max(edge + 1, edge + rem))])
    Pt = np.array([[_c(pm[i] ** (q * TILE_BLOCKS * m_)) for i in range(n8)] for m_ in range(ntiles)])
    bx = np.array([_c(pm[i] ** edge / mp.mpc(modes.kappa[i])) for i in range(n8)])
    # boundary weights c_i p_i^(L-1-n_k), n_k = edge + q k
    bnd = np.zeros((M, n8), dtype=np.complex128)
    rmax = max(abs(v) for v in pm)
    k_bnd = M
    for k in range(M - 1, -1, -1):
        e = L - 1 - (edge + q * k)
        if rmax ** e < mp.mpf(10) ** -30:
            break
        k_bnd = k
        for i in range(n8):
            bnd[k, i] = _c(modes.mp_c[i] * pm[i] ** e)

    Liq = impedance / fs if correct_iq else 0.0
    lam = 1.0 - Liq
    mlam = mp.mpf(1) - mp.mpf(Liq)
    lam_j = np.array([float(mlam ** j) for j in range(q + 1)])
    lam_q = float(mlam ** q)
    lam_N = float(mlam ** N)
    lam_inv = float(1 / mlam)
    lam_k = np.array([float(mlam ** k) for k in range(33)])
    mu_k = np.array([float(mlam ** -k) for k in range(33)])
    RL = -(-Hq // 4)
    run_len = np.zeros(8, dtype=np.int64)
    for k in range(4):
        a0, a1 = min(k * RL, Hq), min((k + 1) * RL, Hq)
        run_len[k] = a1 - a0
        run_len[7 - k] = max(0, (q - a0) - max(q - a1, Hq))   # (a lane past the last pair of an odd block owns nothing)
    assert run_len.sum() == q
    lam_run = np.array([float(mlam ** int(v)) for v in run_len])
    norm = None
    if normalize:
        dom = {'B': (0, 255), 'h': (-32768, 32767), 'b': (-128, 127),
               'i': (-2147483648, 2147483647), 'H': (0, 65536), 'I': (0, 4294967295)}.get(enc)
        if dom is not None:
            norm = (float(dom[0]), 1 / (-dom[0] + dom[1]))

    rows_hz = [int(f) for f in rows_hz]
    R = len(rows_hz)
    w = np.array([reference_w(f, fs) for f in rows_hz])
    # standard mode skips the shift entirely when centre == 0 (dsp_processor.py:185-187);
    # exp(0) == 1 exactly, so a zero phase increment is the same thing.
    use_nco = np.array([bool(simo or f) for f in rows_hz])
    ws = min(q * Mf, N - 1 - edge)
    nend = N - ws
    T2 = np.stack([_phasor(wr, np.arange(q)) for wr in w])
    T3 = np.stack([_phasor(wr, q * np.arange(TILE_BLOCKS + 1)) for wr in w])
    T1 = np.stack([_phasor(wr, q * TILE_BLOCKS * np.arange(ntiles)) for wr in w])
    Ehead = np.stack([_phasor(wr, np.arange(edge + 1)) for wr in w])
    Eend = np.stack([_phasor(wr, ws + np.arange(nend)) for wr in w])

    # IQ corrector, decoupled (see the Plan fields): per-row constants in high precision
    alpha = np.zeros((R, n8), dtype=np.complex128)
    alphaT = np.zeros((R, n8), dtype=np.complex128)
    beta = np.ones((R, n8), dtype=np.complex128)
    betaT = np.ones((R, n8), dtype=np.complex128)
    gamma = np.zeros(R, dtype=np.complex128)
    psiY = np.zeros((2, R, TILE_BLOCKS), dtype=np.complex128)
    phE = _phasor_vec(w, q * Mf)
    lam_tile = np.array([float(mlam ** (q * TILE_BLOCKS)), float(mlam ** (q * cnt_last))])
    if correct_iq:
        g0 = mp.mpf(modes.g0)
        rho = [mp.mpc(v) for v in modes.rho]
        rho_p = [mp.mpc(v) for v in modes.rho_p]
        Lmp = mp.mpf(Liq)
        for r in range(R):
            ejw = mp.expj(mp.mpf(w[r])) if use_nco[r] else mp.mpc(1)
            mu = mlam * ejw                                 # lam * e^{jw}
            dist = min(abs(mu - pm[i]) for i in range(n8))
            if dist < mp.mpf(10) ** -8:
                raise ValueError('the IQ-offset mode lam*e^{jw} coincides with a pole of the decimation '
                                 'filter; shift the centre frequency by 1 Hz')
            a = [1 / (mu - pm[i]) for i in range(n8)]
            aT = [1 / (1 - pm[i] * mu) for i in range(n8)]
            b = [1 + a[i] * Lmp * ejw for i in range(n8)]
            bT = [1 - pm[i] * aT[i] * Lmp * ejw for i in range(n8)]
            gam = sum(rho[i] * a[i] + rho_p[i] * aT[i] for i in range(n8)) + g0
            alpha[r] = [_c(v) for v in a]
            alphaT[r] = [_c(v) for v in aT]
            beta[r] = [_c(v) for v in b]
            betaT[r] = [_c(v) for v in bT]
            gamma[r] = _c(gam)
            muq = mu ** q
            for l in range(TILE_BLOCKS):
                psiY[0, r, l] = psiY[1, r, l] = _c(gam * muq ** l)

    out_sos = None
    if demod in ('fm', 'am'):
        out_sos = np.ascontiguousarray(
            _sig.ellip(3, 1, 30, omega_out, btype='lowpass', analog=False, output='sos',
                       fs=fs // q), dtype=np.float64)
    elif demod in ('usb', 'lsb'):
        # the sideband [0, B] (usb) or [-B, 0] (lsb) Hz: the fm/am output filter's design call at
        # half the width, rotated by +-B/2
        fs_d = fs // q
        if not 0 < omega_out < fs_d / 2:
            raise ValueError(f'{demod}: the sideband width -w {omega_out} Hz must lie strictly between 0 and '
                             f'half the decimated rate ({fs_d} / 2 Hz)')
        out_sos = np.ascontiguousarray(
            _sig.ellip(3, 1, 30, omega_out / 2, btype='lowpass', analog=False, output='sos',
                       fs=fs_d), dtype=np.float64)
    elif demod not in ('re', 'im', 'iq'):          # iq: the complex decimator output, no output low-pass
        raise ValueError(f'Invalid demod type {demod}')
    ssb = {}
    if demod in ('usb', 'lsb'):
        om = ssb_omega(demod, omega_out, fs // q)
        mp.mp.dps = 40
        ssb['ssb_omega'] = om
        ssb['ssb_rot'] = np.array([_c(mp.expj(mp.mpf(om) * k)) for k in range(M + 1)])
    sos_Lseg, sos_AL, sos_CA, sos_AP = 0, None, None, None
    if out_sos is not None:
        sos_Lseg = -(-M // 32)
        mp.mp.dps = 40
        A_, b_, c_, d_ = _cascade_state_space(out_sos)
        ns = A_.rows
        AL = A_ ** sos_Lseg
        sos_AL = np.array([[float(AL[i, j]) for j in range(ns)] for i in range(ns)])
        sos_CA = np.zeros((sos_Lseg, ns))
        cur = c_.copy()
        for i in range(sos_Lseg):
            sos_CA[i] = [float(cur[0, j]) for j in range(ns)]
            cur = cur * A_
        sos_AP = np.zeros((5, ns, ns))
        Apw = AL
        for lv in range(5):
            sos_AP[lv] = [[float(Apw[i, j]) for j in range(ns)] for i in range(ns)]
            Apw = Apw * Apw
    sm = {}
    if seamless:
        D = lookahead_chunks(modes.p, modes.rho_p, N)
        sm['lookahead'] = D
        sm['chunk_step'] = np.array([(f * N) % fs if use_nco[r] else 0 for r, f in enumerate(rows_hz)],
                                    dtype=np.int64)
        sm['PN'] = np.array([[_c(pm[i] ** (N * j)) for i in range(n8)] for j in range(D + 1)])
        if out_sos is not None:
            mp.mp.dps = 40
            A_, b_, c_, d_ = _cascade_state_space(out_sos)
            ns = A_.rows
            AM = A_ ** M
            sm['sos_AM'] = np.array([[float(AM[i, j]) for j in range(ns)] for i in range(ns)])
            # c A^i for i < M: the response of every output of a chunk to the state it starts from
            Af = np.array([[float(A_[i, j]) for j in range(ns)] for i in range(ns)])
            cam = np.zeros((M, ns))
            cur = np.array([float(c_[0, j]) for j in range(ns)])
            blk = sos_Lseg
            for i in range(M):
                if i % blk == 0:           # restart from the exact power every segment
                    cm = c_ * (A_ ** i)
                    cur = np.array([float(cm[0, j]) for j in range(ns)])
                cam[i] = cur
                cur = cur @ Af
            sm['sos_CAM'] = cam
    fm_interp = None
    h = M >> 1
    if demod == 'fm' and not (M == 2 * h and h >= 2 and h & (h - 1) == 0):   # sdrb_api.cu's fft_ok
        # scipy.signal.resample(r, M) is linear in r: its matrix, column by column
        fm_interp = np.ascontiguousarray(_sig.resample(np.eye(h), M, axis=0))
    return Plan(enc=enc, swap=bool(swap), fs=fs, q=q, N=N, edge=edge, L=L, Mf=Mf, rem=rem, M=M,
                ntiles=ntiles, cnt_last=cnt_last, Hq=Hq, rows_hz=rows_hz, R=R, sos=sos, zi=zi,
                modes=modes, P=P, Ec=Ec, Oc=Oc, Ppow=Ppow, Pk=Pk, Pt=Pt, bx=bx, lam_k=lam_k, mu_k=mu_k, bnd=bnd, k_bnd=k_bnd,
                correct_iq=bool(correct_iq), Liq=Liq, lam=lam, lam_j=lam_j, lam_q=lam_q, lam_N=lam_N, lam_inv=lam_inv, RL=RL, run_len=run_len, lam_run=lam_run,
                norm=norm, w=w, use_nco=use_nco, T2=T2, T3=T3, T1=T1, Ehead=Ehead, Eend=Eend,
                ws=ws, nend=nend, alpha=alpha, beta=beta, alphaT=alphaT, betaT=betaT, gamma=gamma, phE=phE, psiY=psiY,
                lam_tile=lam_tile, demod=demod, out_sos=out_sos,
                big_endian_out=bool(simo if big_endian_out is None else big_endian_out),
                fm_interp=fm_interp, sos_Lseg=sos_Lseg, sos_AL=sos_AL, sos_CA=sos_CA, sos_AP=sos_AP,
                seamless=bool(seamless), **sm, **ssb)


# ------------------------------------------------------------------------------------------------
# Tensor-core block front end (k_tc): the block sums AND the block-local part of the outputs as ONE
# exact int8 GEMM over the raw bytes (DESIGN.md 3.4).
#
# Rows of the GEMM are SUPER-BLOCKS of SB = 2 consecutive blocks (K = 2 q sb bytes, 256 or 512).
# Every quantity the epilogue needs from a super-block is a real-linear functional of its integer
# samples -- decode, byte order, the NCO phasor and the modal weights -- i.e. a row of a
# coefficient matrix applied to its bytes.  The coefficients are rounded once to 40-bit fixed
# point (one common binary scale) and cut into ND = 5 balanced base-256 digits; with the raw bytes
# as the other int8 operand every product and every int32 column sum is exact.
#
# Outputs per row of the bank (N slice of Npad = 208 columns), NCOL = 5 digit columns each:
#   o =  0..15  F~_i = sum_j p_i^(2q-1-j) e^{jwj} z_j     (Re, Im interleaved, poles 0..7)
#   o = 16..31  G~_i = sum_j p_i^j e^{jwj} z_j
#   o = 32..35  E_a = sum_{j<q} lam^(q-1-j) z_j,  E_ab = sum_{j<2q} lam^(2q-1-j) z_j   (IQ-EMA aggregates)
#   o = 36..39  yl_a, yl_b: the part of the two block outputs that is local to the super-block
#               (g0 z_0 + sum_i rho'_i betaT_i G~_i  /  sum_i rho_i beta_i F~a_i + rho'_i betaT_i G~b_i + g0 u_q)
#   columns 200.. : x0_a, x0_b = first raw sample of either block, unit coefficients (exact decode
#               check, sdrb_keep_x0), isz columns per component
# 16-bit samples: digit s of a coefficient meets the high byte in column s and the low byte in
# column s+1; the low byte's coefficient is re-rounded to 4 digits (round(A/256)) so that no sixth
# column is needed -- the low byte carries 1/256 of the weight, so its coefficient needs 8 bits
# less for the same absolute error (measured: the chain stays at its FP64 floor).
TC_ND = 5                 # coefficient digits = digit columns per output
TC_SB = 2                 # blocks per GEMM row
TC_NOUT = 40
TC_NPAD = 208
TC_X0COL = 200
TC_NROWC = 200            # complex constants per row for the epilogue (TcTables.rowc)


@dataclass
class TcTables:
    K: int                 # bytes per GEMM row = SB * q * 2 * itemsize
    isz: int               # bytes per I or Q item
    ND: int
    NCOL: int              # digit columns per output (== ND)
    SB: int
    nout: int
    Npad: int
    R: int
    xor_mask: np.ndarray   # (16,) uint8, XOR pattern of one 16-byte group of the raw stream
    a_signed: bool         # the GEMM reads the (fixed-up) raw bytes as signed int8; False: as unsigned
    Bq: np.ndarray         # (R, Npad, K) int8 coefficient digits
    S: int                 # outputs 0..35 are integers * 2^-S
    S_yl: int              # outputs 36..39 (yl_a, yl_b: small coefficients, their own finer scale) * 2^-S_yl
    cst: np.ndarray        # (R, nout + 4) response to the constant the XOR removed (last 4: x0 columns)
    rowc: np.ndarray       # (R, TC_NROWC) complex epilogue constants, see build_tc
    col_l1: int            # max over columns of sum_k |digit|: bounds every int32 column sum


# layout of TcTables.rowc (complex entries)
RC_CA, RC_CB, RC_DA, RC_DB = 0, 8, 16, 24     # output weights on the forward / backward scan states
RC_GAM, RC_GAMQ = 32, 33                      # gamma, gamma e^{jwq}
RC_AGGF = 34                                  # T3x[15]: forward tile aggregate -> tile frame
RC_ROT = 36                                   # [16] T3x[l] = e^{jw 2q l}
RC_POW = 52                                   # [16 modes][9] powers 0..8 of the scan multipliers
RC_END = RC_POW + 16 * 9


def _balanced_digits(A: int, nd: int):
    d = []
    for _ in range(nd):
        r = ((A + 128) % 256) - 128
        d.append(r)
        A = (A - r) // 256
    if A != 0:
        raise OverflowError('coefficient does not fit its digits')
    return d[::-1]


def tc_supported(pl: Plan) -> bool:
    """Shapes the tensor-core front end handles; everything else takes the FP64 block kernel."""
    if pl.enc not in ('b', 'B', 'h', 'H') or pl.norm is not None:
        return False
    K = TC_SB * pl.q * 2 * _ITEMSIZE[pl.enc]
    return (K in (256, 512) and pl.rem == 0 and pl.Mf % TILE_BLOCKS == 0
            and (pl.Mf // TC_SB) % 128 == 0 and 1 <= pl.R <= 32 and pl.q >= pl.edge + 1)


def build_tc(pl: Plan, nd: int = TC_ND) -> TcTables | None:
    if not tc_supported(pl):
        return None
    _heavy()
    mp.mp.dps = 50
    q, R = pl.q, pl.R
    q2 = TC_SB * q
    isz = _ITEMSIZE[pl.enc]
    sb = 2 * isz
    K = q2 * sb
    signed = pl.enc in ('b', 'h')
    stored_le = not pl.swap
    ncol = nd
    nout = TC_NOUT
    pm = pl.modes.mp_p
    lam = mp.mpf(1) - mp.mpf(pl.Liq)
    g0 = mp.mpf(pl.modes.g0)
    rho = [mp.mpc(v) for v in pl.modes.rho]
    rho_p = [mp.mpc(v) for v in pl.modes.rho_p]
    # pole powers p_i^n, n <= 2q: the same for every row of the bank (most of the build time otherwise)
    pw = [[pm[i] ** n for n in range(q2 + 1)] for i in range(8)]

    # byte bookkeeping of one sample: (component, significance) per byte
    info = []
    for bb in range(sb):
        cpt, bi = divmod(bb, isz)
        info.append((cpt, bi if stored_le else isz - 1 - bi))

    allrows = []   # [r][o] -> list over j of (coef on I_j, coef on Q_j), real mp numbers
    rowc = np.zeros((R, TC_NROWC), dtype=np.complex128)
    for r in range(R):
        rows = []
        if pl.use_nco[r]:
            T2x = [mp.mpc(complex(v)) for v in _phasor(pl.w[r], np.arange(q2))]
        else:
            T2x = [mp.mpc(1)] * q2
        rb = [rho[i] * mp.mpc(complex(pl.beta[r, i])) for i in range(8)]
        rbT = [rho_p[i] * mp.mpc(complex(pl.betaT[r, i])) for i in range(8)]
        cplx = []
        for i in range(8):
            cplx.append([pw[i][q2 - 1 - j] * T2x[j] for j in range(q2)])
        for i in range(8):
            cplx.append([pw[i][j] * T2x[j] for j in range(q2)])
        for c in cplx:
            rows.append([(mp.re(v), -mp.im(v)) for v in c])    # Re(c*(I+jQ)) = cr I - ci Q
            rows.append([(mp.im(v), mp.re(v)) for v in c])     # Im(c*(I+jQ)) = ci I + cr Q
        ea = [lam ** (q - 1 - j) if j < q else mp.mpf(0) for j in range(q2)]
        eab = [lam ** (q2 - 1 - j) for j in range(q2)]
        for e in (ea, eab):
            rows.append([(v, mp.mpf(0)) for v in e])
            rows.append([(mp.mpf(0), v) for v in e])
        yla = [sum(rbT[i] * pw[i][j] for i in range(8)) * T2x[j] + (g0 if j == 0 else 0) for j in range(q2)]
        ylb = []
        for j in range(q2):
            if j < q:
                ylb.append(sum(rb[i] * pw[i][q - 1 - j] for i in range(8)) * T2x[j])
            else:
                ylb.append((sum(rbT[i] * pw[i][j - q] for i in range(8)) + (g0 if j == q else 0)) * T2x[j])
        for c in (yla, ylb):
            rows.append([(mp.re(v), -mp.im(v)) for v in c])
            rows.append([(mp.im(v), mp.re(v)) for v in c])
        allrows.append(rows)

        # ---- epilogue constants of this row (k_tc: tc_epilogue; tests/emulator.py: emu_main_tc)
        eps2 = T2x[q] * T2x[q]                                 # e^{jw 2q}
        P2 = [pw[i][q2] for i in range(8)]
        Pq = [pw[i][q] for i in range(8)]
        ce = mp.conj(eps2)
        for i in range(8):
            rowc[r, RC_CA + i] = _c(rb[i] * ce)                # y_a += ca_i A_i
            rowc[r, RC_CB + i] = _c(rbT[i] * P2[i] * eps2)     # y_a += cb_i B_i
            rowc[r, RC_DA + i] = _c(rb[i] * Pq[i] * ce)        # y_b += da_i A_i
            rowc[r, RC_DB + i] = _c(rbT[i] * Pq[i] * eps2)     # y_b += db_i B_i
        gam = mp.mpc(complex(pl.gamma[r]))
        rowc[r, RC_GAM] = _c(gam)
        rowc[r, RC_GAMQ] = _c(gam * T2x[q])
        for l in range(16):
            rowc[r, RC_ROT + l] = _c(eps2 ** l)
        rowc[r, RC_AGGF] = _c(eps2 ** 15)
        for i in range(8):
            for k in range(9):
                rowc[r, RC_POW + i * 9 + k] = _c((ce * P2[i]) ** k)            # forward scan multiplier
                rowc[r, RC_POW + (8 + i) * 9 + k] = _c((eps2 * P2[i]) ** k)    # backward

    # one binary scale for the modal sums and E of every row, a finer one for the local outputs
    # (their coefficients are ~1/75 of the modal ones and enter y with weight 1, not rho)
    lim = 127 * 256 ** (nd - 1)
    amax = max(max(abs(a), abs(b)) for rows in allrows for row in rows[:36] for a, b in row)
    ayl = max(max(abs(a), abs(b)) for rows in allrows for row in rows[36:] for a, b in row)
    S_hi = [int(mp.floor(mp.log(lim / amax, 2))), int(mp.floor(mp.log(lim / ayl, 2)))]   # top-byte coefficient = round(c 2^S_hi)
    S, S_yl = (v - 8 * (isz - 1) for v in S_hi)       # output integer V = value * 2^S

    Bq = np.zeros((R, TC_NPAD, K), dtype=np.int8)
    for r in range(R):
        for o, row in enumerate(allrows[r]):
            c0 = ncol * o
            for j, ab in enumerate(row):
                for cpt in (0, 1):
                    A = int(mp.nint(ab[cpt] * mp.mpf(2) ** S_hi[o >= 36]))
                    for bb, (c2_, w) in enumerate(info):
                        if c2_ != cpt:
                            continue
                        if w == isz - 1:                       # top (or only) byte: all nd digits
                            for s_, dv in enumerate(_balanced_digits(A, nd)):
                                Bq[r, c0 + s_, j * sb + bb] = dv
                        else:                                  # low byte: re-rounded, one digit less
                            Alo = (A + 128) // 256
                            for s_, dv in enumerate(_balanced_digits(Alo, nd - 1)):
                                Bq[r, c0 + 1 + s_, j * sb + bb] = dv
        # x0_a, x0_b: first sample of either block, exact (coefficient 1 on its own bytes)
        for blk in (0, 1):
            for cpt in (0, 1):
                c0 = TC_X0COL + (2 * blk + cpt) * isz
                for bb, (c2_, w) in enumerate(info):
                    if c2_ == cpt:
                        Bq[r, c0 + (isz - 1 - w), blk * q * sb + bb] = 1
    # Signedness.  The tensor core reads the whole A operand either as signed or as unsigned int8.
    # Unsigned 8-bit samples go in as they are when the int32 digit-pair sums are provably safe for
    # bytes up to 255 (K = 256); 'b' goes in as it is (signed).  Everything else takes the signed
    # route: the bytes that are not a signed top byte are XOR-ed with 0x80 (u -> u - 128 as int8) by
    # the kernel's sign fix-up warps, and the response to the constant this removes is added back.
    col_l1 = int(np.abs(Bq.astype(np.int64)).sum(axis=2).max())
    a_signed = not (pl.enc == 'B' and col_l1 * 255 * 257 < 2 ** 31)
    xflag = [a_signed and not (signed and w == isz - 1) for (_c, w) in info]
    xor_mask = np.array([0x80 if xflag[b % sb] else 0 for b in range(16)], dtype=np.uint8)
    xk = np.array([128 if xflag[k % sb] else 0 for k in range(K)], dtype=np.int64)
    colsum = Bq.astype(np.int64) @ xk                                  # (R, Npad)
    cst = np.zeros((R, nout + 4))
    for r in range(R):
        for o in range(nout):
            V = 0
            for t in range(ncol):
                V = V * 256 + int(colsum[r, ncol * o + t])
            cst[r, o] = float(mp.mpf(V) * mp.mpf(2) ** (-(S_yl if o >= 36 else S)))
        for x in range(4):
            V = 0
            for t in range(isz):
                V = V * 256 + int(colsum[r, TC_X0COL + x * isz + t])
            cst[r, nout + x] = float(V)
    amax_byte = 128 if a_signed else 255
    if col_l1 * amax_byte * 257 >= 2 ** 31:
        raise OverflowError('int32 digit-pair sums could overflow for this coefficient set')
    return TcTables(K=K, isz=isz, ND=nd, NCOL=ncol, SB=TC_SB, nout=nout, Npad=TC_NPAD, R=R, xor_mask=xor_mask,
                    a_signed=a_signed,
                    Bq=Bq, S=S, S_yl=S_yl, cst=cst, rowc=rowc, col_l1=col_l1)


# ------------------------------------------------------------------------------------------------
def build_tc_or_none(pl: Plan) -> TcTables | None:
    """``build_tc`` for the shapes it takes; a coefficient set whose int32 digit sums could overflow
    (not seen: the worst of the swept frequencies uses 54 % of the range) is left to the FP64 block
    kernel instead of failing the run."""
    try:
        return build_tc(pl)
    except OverflowError:
        return None


def cache_dir() -> str:
    import os
    return os.environ.get('SDRB_PLAN_CACHE', os.path.join(os.path.dirname(os.path.abspath(__file__)), '.plan_cache'))


def cached_plan(*args, **kwargs):
    """``(build_plan(*args, **kwargs), build_tc(plan))`` through an on-disk cache (directory
    ``$SDRB_PLAN_CACHE``, default ``.plan_cache`` next to this package; set it to an empty string
    to switch the cache off; an unwritable directory simply means no caching).  The tables depend only on the arguments and on this file, so the key is their
    hash; building them takes seconds of 50-digit arithmetic, which matters to a command-line run
    and to nothing else."""
    import hashlib
    import os
    import pickle
    root = cache_dir()
    path = None
    if root:
        with open(__file__, 'rb') as fh:
            ver = hashlib.sha256(fh.read()).hexdigest()[:16]
        key = hashlib.sha256(repr((args, sorted(kwargs.items()), ver)).encode()).hexdigest()[:32]
        path = os.path.join(root, f'plan_{key}.pkl')
        try:
            with open(path, 'rb') as fh:
                return pickle.load(fh)
        except Exception:
            pass
    pl = build_plan(*args, **kwargs)
    tc = build_tc_or_none(pl)
    pl.modes.mp_p = pl.modes.mp_c = None              # high-precision scratch of the build, not part of the plan
    if path:
        try:
            os.makedirs(root, exist_ok=True)
            tmp = f'{path}.{os.getpid()}.tmp'
            with open(tmp, 'wb') as fh:
                pickle.dump((pl, tc), fh, protocol=pickle.HIGHEST_PROTOCOL)
            os.replace(tmp, path)
        except OSError:
            pass
    return pl, tc
