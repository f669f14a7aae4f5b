"""Single-sideband output (``-m usb`` / ``-m lsb``) without a GPU: the oracle (against a direct
convolution and its selectivity), a numpy twin of the kernels' segmented complex filter, the plan's
tables against the rotated recurrence, the refusals, the C-ABI constants and the host layers."""
import json
import os
import pickle
import re

import numpy as np
import pytest
from scipy import signal

from oracle import oracle as orc
from sdrterm_b200 import _native as nat
from sdrterm_b200.plan import _cascade_state_space, _heavy, build_plan
from ssb_ref import ssb, ssb_omega, ssb_oracle, ssb_sos

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS, Q, B = 1_024_000, 64, 3000
FSD = FS // Q


def _y(n, seed=1):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(n) + 1j * rng.standard_normal(n)


def _state_space(sos):
    _heavy()
    from sdrterm_b200 import plan as P
    P.mp.mp.dps = 40
    A, b, c, d = _cascade_state_space(sos)
    f = lambda m: np.array([[float(m[i, j]) for j in range(m.cols)] for i in range(m.rows)])
    return f(A), f(b)[:, 0], f(c)[0], float(d)


@pytest.mark.parametrize('demod', ['usb', 'lsb'])
def test_oracle_is_the_complex_band_pass(demod):
    """Re of the convolution with the truncated complex impulse response h[m] e^{j Omega m}."""
    sos, om = ssb_sos(FS, Q, B), ssb_omega(demod, B, FSD)
    y = _y(3000)
    h = signal.sosfilt(sos, np.r_[1.0, np.zeros(2999)])
    hb = h * np.exp(1j * om * np.arange(h.size))
    ref = np.real(np.convolve(y, hb)[:y.size])
    assert np.max(np.abs(ssb(y, sos, om) - ref)) < 1e-12 * np.max(np.abs(ref))


@pytest.mark.parametrize('f,keep', [(B / 2, 'usb'), (-B / 2, 'lsb')])
def test_oracle_selects_one_sideband(f, keep):
    sos = ssb_sos(FS, Q, B)
    k = np.arange(8000)
    y = np.exp(2j * np.pi * f / FSD * k)
    for demod in ('usb', 'lsb'):
        s = ssb(y, sos, ssb_omega(demod, B, FSD))[4000:]          # settled
        level = 20 * np.log10(np.max(np.abs(s)))
        if demod == keep:
            assert -1.0 - 1e-9 <= level <= 1e-9
        else:
            assert level <= -30.0


def test_lsb_of_the_conjugate_is_usb():
    sos, y = ssb_sos(FS, Q, B), _y(2048, 3)
    a = ssb(np.conj(y), sos, ssb_omega('lsb', B, FSD))
    b = ssb(y, sos, ssb_omega('usb', B, FSD))
    assert np.max(np.abs(a - b)) <= 1e-13 * np.max(np.abs(b))


def _segmented_twin(y, pl):
    """The kernels' decomposition (k_finish / k_seam_demod): lane segments of Lseg outputs in the
    Weaver frame from a zero state, the Kogge-Stone scan of the segment maps with (A^Lseg)^(2^lv),
    every output then gets c A^j s_in; s = Re(e^{j Omega k} v)."""
    M, Ls = y.size, pl.sos_Lseg
    rot = pl.ssb_rot[:M]
    u = y * np.conj(rot)
    v = np.zeros(M, dtype=np.complex128)
    ends = np.zeros((32, 4), dtype=np.complex128)
    for g in range(32):
        seg = u[g * Ls:(g + 1) * Ls]
        v[g * Ls:(g + 1) * Ls], zf = signal.sosfilt(pl.out_sos, seg, zi=np.zeros((2, 2), dtype=np.complex128))
        ends[g] = zf.reshape(-1)
    st = ends.copy()
    for lv in range(5):
        sh = 1 << lv
        prev = st.copy()
        for g in range(sh, 32):
            st[g] = pl.sos_AP[lv] @ prev[g - sh] + prev[g]
    sin = np.vstack([np.zeros(4), st[:-1]])
    for g in range(32):
        v[g * Ls:(g + 1) * Ls] += pl.sos_CA @ sin[g]
    return np.real(rot * v)


@pytest.mark.parametrize('demod', ['usb', 'lsb'])
def test_segmented_twin_matches_oracle(demod):
    pl = build_plan(FS, 'h', Q, [15000], demod=demod, omega_out=B)
    y = _y(pl.M, 5)
    ref = ssb(y, pl.out_sos, pl.ssb_omega)
    assert np.max(np.abs(_segmented_twin(y, pl) - ref)) < 1e-12 * np.max(np.abs(ref))


@pytest.mark.parametrize('demod', ['usb', 'lsb'])
def test_tables_against_the_rotated_recurrence(demod):
    """The complex segment map A'^Lseg, the seamless chunk map A'^M and c'A'^k of the rotated
    prototype (e^{j Omega} A, e^{j Omega} b, c, d), by brute force, against the real tables times the
    plan's rotations; and the rotated recurrence itself against the oracle."""
    pl = build_plan(FS, 'h', Q, [15000], demod=demod, omega_out=B, seamless=True)
    assert pl.ssb_omega == pytest.approx(ssb_omega(demod, B, FSD), rel=1e-15)
    assert np.allclose(pl.ssb_rot, np.exp(1j * pl.ssb_omega * np.arange(pl.M + 1)), rtol=0, atol=1e-13)
    A, b, c, d = _state_space(pl.out_sos)
    e = np.exp(1j * pl.ssb_omega)
    Ar = e * A
    P = np.eye(4, dtype=np.complex128)
    cur = c.astype(np.complex128)
    for k in range(pl.M):
        if k < pl.sos_Lseg:
            assert np.max(np.abs(cur - pl.ssb_rot[k] * pl.sos_CA[k])) < 1e-13
        assert np.max(np.abs(cur - pl.ssb_rot[k] * pl.sos_CAM[k])) < 1e-12
        if k == pl.sos_Lseg:
            assert np.max(np.abs(P - pl.ssb_rot[k] * pl.sos_AL)) < 1e-13
        cur = cur @ Ar
        P = Ar @ P
    assert np.max(np.abs(P - pl.ssb_rot[pl.M] * pl.sos_AM)) < 1e-12
    y = _y(700, 9)
    s = np.zeros(4, dtype=np.complex128)
    out = np.empty(y.size)
    for k, x in enumerate(y):
        out[k] = np.real(c @ s + d * x)
        s = Ar @ s + e * b * x
    ref = ssb(y, pl.out_sos, pl.ssb_omega)
    assert np.max(np.abs(out - ref)) < 1e-12 * np.max(np.abs(ref))


def test_plan_ssb_tables_and_width():
    pl = build_plan(FS, 'h', Q, [15000], correct_iq=True, demod='usb', omega_out=B)
    assert pl.W == pl.M == 512 and pl.out_sos.shape == (2, 6) and pl.sos_AP.shape == (5, 4, 4)
    assert np.array_equal(pl.out_sos, ssb_sos(FS, Q, B))
    assert nat.DEMOD_CODE['usb'] == nat.USB == 5 and nat.DEMOD_CODE['lsb'] == nat.LSB == 6
    ragged = build_plan(2_400_000, 'B', 50, [0], demod='lsb', omega_out=10000)
    assert ragged.M == ragged.W == 1311 and ragged.ssb_rot.shape == (1312,) and ragged.ssb_omega < 0


@pytest.mark.parametrize('w', [0, -100, FSD // 2, FSD])
def test_refuses_a_sideband_outside_the_band(w):
    for demod in ('usb', 'lsb'):
        with pytest.raises(ValueError):
            build_plan(FS, 'h', Q, [15000], demod=demod, omega_out=w)
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    p = DspProcessor(FS, center=15000, omegaOut=w, dec=Q, enc='h')
    with pytest.raises(ValueError):
        p.selectOutputUsb()
    with pytest.raises(ValueError):
        p.selectOutputLsb()


def test_refuses_seamless_without_whole_blocks_and_smoothing_with_seamless():
    with pytest.raises(ValueError):
        build_plan(2_400_000, 'B', 50, [0], demod='usb', omega_out=10000, seamless=True)
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    with pytest.raises(ValueError):
        DspProcessor(FS, center=15000, omegaOut=B, dec=Q, enc='h', smooth=True, seamless=True)


def test_header_constants_match_python():
    src = open(os.path.join(ROOT, 'include', 'sdrterm_b200.h')).read()
    m = re.search(r'enum sdrb_demod \{([^}]*)\}', src)
    consts = dict((k, int(v)) for k, v in re.findall(r'(SDRB_\w+) = (\d+)', m.group(1)))
    assert consts['SDRB_USB'] == nat.USB and consts['SDRB_LSB'] == nat.LSB
    assert int(re.search(r'#define SDRB_ABI_VERSION (\d+)', src).group(1)) == nat.ABI_VERSION == 11
    assert 'sdrb_ssb_demod' in nat.EXPORTS and 'int sdrb_ssb_demod(' in src
    assert [f[0] for f in nat.Tables._fields_][-2:] == ['ssb_omega', 'ssb_rot']


def test_cli_and_selectors():
    from sdrterm_b200.dsp import demodulation as dem
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    from sdrterm_b200.dsp.vfo_processor import VfoProcessor
    from sdrterm_b200.misc import file_util
    from sdrterm_b200.misc.io_args import DemodulationChoices, selectDemodulation
    from sdrterm_b200.sdrterm import buildParser, makeProcessor
    a = buildParser().parse_args(['-r', '1024k', '-c', '15k', '-d', '64', '-e', 'h', '-m', 'USB', '-w', '3k'])
    assert a.demod == 'usb' and a.omegaOut == 3000
    p = makeProcessor(a, file_util.parseRawType(None, a.fs, a.enc))
    assert isinstance(p, DspProcessor) and p.demod == dem.usbDemod and p.bandwidth == 3000
    assert p._demodName() == 'usb' and np.allclose(p._outputFilters, ssb_sos(FS, Q, 3000))
    b = buildParser().parse_args(['-r', '2400k', '-e', 'h', '--simo', '--vfos', '100000', '-d', '64', '-m', 'lsb',
                                  '-w', '5000', '--vfo-host', '127.0.0.1:0'])
    v = makeProcessor(b, file_util.parseRawType(None, b.fs, b.enc))
    assert isinstance(v, VfoProcessor) and v.demod == dem.lsbDemod and v._demodName() == 'lsb' and v.bandwidth == 5000
    assert str(DemodulationChoices.USB) == 'usb' and str(DemodulationChoices.LSB) == 'lsb'
    q = DspProcessor(48000, omegaOut=3000)
    selectDemodulation(DemodulationChoices.LSB, q)()
    assert q.demod == dem.lsbDemod
    selectDemodulation('usb', q)()
    assert q.demod == dem.usbDemod


@pytest.mark.parametrize('demod', ['usb', 'lsb'])
def test_pickle_and_repr_keep_the_mode(demod):
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    p = DspProcessor(FS, center=15000, omegaOut=B, dec=Q, enc='h', correctIq=True)
    getattr(p, 'selectOutput' + demod.capitalize())()
    q = pickle.loads(pickle.dumps(p))
    assert q._demodName() == demod and q._engine is None and q.bandwidth == B
    d = json.loads(repr(q))
    assert d['demodulation'] == demod and d['omegaOut'] == B
    p.selectOutputFm()
    assert 'demodulation' not in json.loads(repr(p))


def test_operator_checks_its_arguments():
    from sdrterm_b200.dsp import demodulation as dem
    with pytest.raises(ValueError):
        dem.ssbDemod(np.zeros((1, 8), dtype=np.complex128), np.zeros((1, 9)), ssb_sos(FS, Q, B), 0.5)
    with pytest.raises(ValueError):
        dem.usbDemod(np.zeros((1, 8), dtype=np.complex128), np.zeros((1, 8)), ssb_sos(FS, Q, B), -0.5)
    with pytest.raises(ValueError):
        dem.lsbDemod(np.zeros((1, 8), dtype=np.complex128), np.zeros((1, 8)), ssb_sos(FS, Q, B), 0.5)


def test_cached_plan_keeps_modes_apart(tmp_path, monkeypatch):
    from sdrterm_b200.plan import cached_plan
    monkeypatch.setenv('SDRB_PLAN_CACHE', str(tmp_path))
    args = (2_400_000, 'f', 64, [30000])
    seen = {}
    for demod in ('usb', 'lsb', 'usb', 'fm'):
        pl, tc = cached_plan(*args, demod=demod, omega_out=5000)
        assert pl.demod == demod and pl.W == pl.M
        if demod != 'fm':
            seen.setdefault(demod, pl.ssb_rot)
            assert np.array_equal(seen[demod], pl.ssb_rot)
        else:
            assert pl.ssb_rot is None
    assert np.allclose(seen['usb'], np.conj(seen['lsb']), rtol=0, atol=1e-15)
    assert len(list(tmp_path.glob('plan_*.pkl'))) == 3

