"""GPU parity at the shapes round 1 never compared with the oracle (VERDICT r1, "what's weak" 1-4):
BASELINE config 4 at its real width (256 VFOs + centre, float32), the R = 32 / R = 33 boundary
between the tensor-core and the FP64 block front ends, the double-buffered ``sdrb_submit`` /
``sdrb_wait`` host path with alternating slots, and the integer decode bit for bit.
Tolerance as everywhere: max|out - ref| / max|ref| <= 1e-9 (BASELINE.json north_star)."""
import numpy as np
import pytest

import signals
from oracle import oracle as orc
from util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-9
CB = 131072


def _simo_kw(fs, enc, vfos, swap, demod='fm', omega=5000, dec=64):
    return dict(fs=fs, enc=enc, center=0, dec=dec, demod=demod, omega_out=omega, correct_iq=False,
                vfos=vfos, simo=True, normalize=False, swap=swap, big_endian=None)


def test_config4_full_width_257_rows_float32():
    """BASELINE config 4: 61.44 MS/s float32 IQ, 256 VFOs on a 200 kHz grid + the centre = 257
    rows, FM, -d 64, big-endian doubles per row (SURVEY 8d table, 8-Q3: FP64 chain on the widened
    float32 samples)."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    body, vfos = signals.c4_bytes(2 * 16384, seed=4, k=256)
    kw = _simo_kw(61_440_000, 'f', vfos, False, omega=12500)
    pl = plan_for(kw)
    assert pl.R == 257 and pl.M == 256
    with Engine(pl, max_chunks=2, keep_decimated=True) as eng:
        out = eng.process(body)
        y = eng.decimated(2)
    ch = orc.Chain(**kw, nthreads=orc.max_threads())
    ref = ch.run_fast(body)
    assert out.dtype == np.dtype('>f8') and out.shape == ref.shape == (257, 2 * 256)
    assert rel_err(np.asarray(out, dtype=np.float64), ref) < TOL
    # every row individually (a row-indexing slip would hide in the global maximum)
    got = np.asarray(out, dtype=np.float64)
    for r in (0, 1, 127, 128, 255, 256):
        assert rel_err(got[r], ref[r]) < TOL, r
    assert np.isfinite(y).all()


@pytest.mark.parametrize('k', [31, 32, 33])
def test_row_count_boundary_between_front_ends(k):
    """k VFOs + centre: 32 rows is the widest bank the tensor-core front end takes, 33 and 34 go
    to the FP64 block kernel; all three against the oracle, int16 big-endian as config 3."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    body, vfos = signals.c3_bytes(2 * 32768, seed=3, k=k, step=30_000)
    kw = _simo_kw(2_400_000, 'h', vfos, True)
    pl = plan_for(kw)
    assert pl.R == k + 1
    with Engine(pl, max_chunks=2) as eng:
        assert (eng.tc is not None) == (pl.R <= 32)
        out = eng.process(body)
    ref = orc.Chain(**kw, nthreads=orc.max_threads()).run_fast(body)
    got = np.asarray(out, dtype=np.float64)
    assert got.shape == ref.shape
    assert rel_err(got, ref) < TOL
    for r in range(pl.R):
        assert rel_err(got[r], ref[r]) < TOL, r


@pytest.mark.parametrize('sub', [3, 5])
def test_submit_wait_alternating_slots_with_iq_state(sub):
    """The timed end-to-end path of bench.py: >= 6 batches through sdrb_submit / sdrb_wait with the
    two slots alternating (H2D of batch i+1 overlaps the kernels of batch i; the scratch and the
    IQ-corrector state are shared between the slots), pinned host buffers, --correct-iq on;
    the concatenation equals the oracle over the whole stream."""
    import torch
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    nch = 6 * sub + 2                                     # a short last batch as well
    body = signals.c1_bytes(nch * 32768, seed=21, header=False)
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=False, big_endian=None)
    pl = plan_for(kw)
    host_raw = torch.frombuffer(bytearray(body), dtype=torch.uint8).pin_memory()
    nb = -(-nch // sub)
    host_out = [torch.empty(sub * pl.M, dtype=torch.float64).pin_memory() for _ in range(2)]
    parts = []
    with Engine(pl, max_chunks=sub) as eng:
        pend = [None, None]
        for b in range(nb):
            s = b & 1
            if pend[s] is not None:
                eng.wait(s)
                parts.append((pend[s][0], host_out[s][:pend[s][1] * pl.M].clone()))
            n = min(sub, nch - b * sub)
            eng.submit(s, host_raw.data_ptr() + b * sub * CB, n, host_out[s].data_ptr())
            pend[s] = (b, n)
        for s in ((nb & 1), ((nb + 1) & 1)):              # older batch first
            if pend[s] is not None:
                eng.wait(s)
                parts.append((pend[s][0], host_out[s][:pend[s][1] * pl.M].clone()))
        off = eng.iq_state
    parts.sort(key=lambda t: t[0])
    got = torch.cat([p for _, p in parts]).numpy()[None]
    ch = orc.Chain(**kw, nthreads=orc.max_threads())
    ref = ch.run_fast(body)
    assert got.shape == ref.shape
    assert rel_err(got, ref) < TOL
    assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))


@pytest.mark.parametrize('enc', ['b', 'B', 'h', 'H', 'i', 'I', 'f', 'd'])
@pytest.mark.parametrize('swap', [False, True])
def test_decode_is_bit_exact(enc, swap):
    """read_file.py:100-101 (`re + 1j*im` on the structured view) on the device, every encoding
    and both byte orders, including the extreme values: array_equal, not a tolerance."""
    from sdrterm_b200.misc.read_file import decodeIq
    rng = np.random.default_rng(5)
    dt = np.dtype({'b': 'i1', 'B': 'u1', 'h': 'i2', 'H': 'u2', 'i': 'i4', 'I': 'u4', 'f': 'f4', 'd': 'f8'}[enc])
    n = 4096
    if dt.kind in 'iu':
        info = np.iinfo(dt)
        v = rng.integers(info.min, info.max, size=2 * n, endpoint=True, dtype=dt)
        v[:4] = [info.min, info.max, info.min, info.max]
    else:
        v = rng.standard_normal(2 * n).astype(dt)
        v[:4] = [np.finfo(dt).max, -np.finfo(dt).tiny, 0.0, -0.0]
    stored = v.astype(dt.newbyteorder('>' if swap else '<'))
    got = decodeIq(stored.tobytes(), enc, swap)
    ref = v[0::2].astype(np.float64) + 1j * v[1::2].astype(np.float64)
    assert got.dtype == np.complex128 and np.array_equal(got, ref)


@pytest.mark.parametrize('enc,swap', [('b', False), ('B', False), ('h', False), ('h', True), ('H', False), ('H', True)])
def test_tensor_core_front_end_decodes_exactly(enc, swap):
    """The tensor-core front end never decodes: the raw bytes are the int8 GEMM operand.  Its two
    unit-coefficient outputs per block (`x0`, the block's first sample) come back through
    sdrb_read_x0 and must equal numpy's decode exactly -- this pins the sign fix-up (XOR 0x80 and
    its constant), the byte order, the TMA layout and the digit recombination."""
    from sdrterm_b200.engine import Engine
    from sdrterm_b200.plan import build_plan
    rng = np.random.default_rng(9)
    isz = 1 if enc in 'bB' else 2
    dt = np.dtype({'b': 'i1', 'B': 'u1', 'h': 'i2', 'H': 'u2'}[enc])
    N = CB // (2 * isz)
    nch = 3
    info = np.iinfo(dt)
    v = rng.integers(info.min, info.max, size=2 * N * nch, endpoint=True, dtype=dt)
    v[:2] = [info.min, info.max]
    stored = v.astype(dt.newbyteorder('>' if swap else '<'))
    q = 64
    pl = build_plan(1_000_000, enc, q, [12_345], swap=swap, correct_iq=True, demod='re')
    with Engine(pl, max_chunks=nch, keep_x0=True) as eng:
        assert eng.tc is not None
        eng.process(stored.tobytes())
        x0 = eng.block_first_samples(nch)                 # (nch, R, Mf) complex
    z = v[0::2].astype(np.float64) + 1j * v[1::2].astype(np.float64)
    ref = z.reshape(nch, N)[:, ::q]
    assert x0.shape == (nch, 1, N // q)
    assert np.array_equal(x0[:, 0, :], ref)


@pytest.mark.parametrize('use_tc', [True, False])
def test_simo_bank_with_iq_correction(use_tc):
    """--simo together with --correct-iq: the decoupled corrector's per-row constants (alpha, beta,
    gamma depend on each row's NCO frequency) on both front ends and in the fused finish kernel's
    R > 1 path; no BASELINE config combines the two, so no golden case does either."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    # one FM carrier per row (a row that held only noise would make the FM output ill-conditioned:
    # the phase of a near-zero pair product), a DC offset for the corrector to remove
    fs, n = 1_024_000, 3 * 32768
    rng = np.random.default_rng(31)
    z = np.zeros(n, dtype=np.complex128)
    for i, f in enumerate((-5000, 22000, 46000, 15000)):
        z += signals._fm_carrier(n, fs, f, 800 + 50 * i, 2000, 3000.0, phase0=0.4 * i)
    z += rng.normal(0, 100, n) + 1j * rng.normal(0, 100, n) + (37 - 21j)
    body = signals._interleave(z, '<i2', -32768, 32767).tobytes()
    kw = dict(fs=fs, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True,
              vfos='-20000,7000,31000', simo=True, normalize=False, swap=False, big_endian=None)
    pl = plan_for(kw)
    assert pl.R == 4 and np.abs(pl.gamma).min() >= 0
    with Engine(pl, max_chunks=3, use_tc=use_tc) as eng:
        assert (eng.tc is not None) == use_tc
        out = eng.process(body)
        off = eng.iq_state
    ch = orc.Chain(**kw)
    ref = ch.run(body)
    got = np.asarray(out, dtype=np.float64)
    assert got.shape == ref.shape
    for r in range(pl.R):
        assert rel_err(got[r], ref[r]) < TOL, r
    assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))


@pytest.mark.parametrize('enc,q,swap', [('b', 128, False), ('B', 128, False), ('h', 32, True), ('H', 64, False)])
def test_tensor_core_shapes_not_covered_by_the_golden_cases(enc, q, swap):
    """K = 512 with 8-bit samples (q = 128), K = 256 with 16-bit samples (q = 32), unsigned 16-bit
    at q = 64: FM with IQ correction against the oracle."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    isz = 1 if enc in 'bB' else 2
    n = 2 * (CB // (2 * isz))
    body = signals.generic_bytes(enc, n, 41, 1_000_000, 30_000, big_endian=swap)
    kw = dict(fs=1_000_000, enc=enc, center=30000, dec=q, demod='fm', omega_out=3000, correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=swap, big_endian=None)
    pl = plan_for(kw)
    with Engine(pl, max_chunks=2) as eng:
        assert eng.tc is not None and eng.tc.K == 2 * q * 2 * isz
        out = eng.process(body)
    ref = orc.Chain(**kw).run(body)
    assert out.shape == ref.shape and rel_err(out, ref) < TOL


def test_file_sharded_entry_point_single_process(tmp_path):
    """multigpu.run_file_sharded (BASELINE config 5's product entry point) with world = 1: a raw
    int16 file whose size is not a whole number of chunks (stale tail, SURVEY 8-Q5), processed in
    batches of 2 chunks, equals the oracle over the same stream."""
    import torch
    from sdrterm_b200 import multigpu
    body = signals.c1_bytes(5 * 32768 + 7000, seed=17, header=False)
    path = tmp_path / 'in.raw'
    path.write_bytes(body)
    out = multigpu.run_file_sharded(str(path), None, fs=1_024_000, enc='h', dec=64, center=15000, omega_out=5000,
                                    correct_iq=True, batch_chunks=2, device=0, dist=None, torch=torch)
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=False, big_endian=None)
    ref = orc.Chain(**kw).run(body)
    assert out.shape == ref.shape and rel_err(out, ref) < TOL


@pytest.mark.parametrize('enc,q,demod,iq,norm,center', [
    ('h', 5, 'am', True, False, 30000),      # odd block: a middle sample without a mirror
    ('B', 25, 'am', True, True, 0),          # odd, normalised input (a normalised zero is not zero), no NCO
    ('f', 63, 'fm', False, False, -20000),   # odd, float32, 4*RL > ceil(q/2): empty pair slots
    ('b', 3, 're', True, False, 10000),      # the smallest odd block
    ('i', 50, 'fm', True, False, 15000),     # even but ragged (rem != 0), 32-bit integers
    ('d', 10, 'am', False, False, 5000),     # float64 samples (16 bytes per sample)
    ('h', 200, 're', True, False, 20000),    # rem = 168: the IQ-corrected end window runs in rounds of 32
])
def test_fp64_block_kernel_odd_and_ragged_blocks(enc, q, demod, iq, norm, center):
    """k_main keeps the raw tile in fragment order (sample j beside its mirror q-1-j, DESIGN 3.5):
    odd q leaves the middle sample alone in its slot, q with 4*ceil(ceil(q/2)/4) > ceil(q/2) leaves
    whole slots empty, and a ragged chunk ends in a partial block.  None of the golden cases has an
    odd q; the oracle handles any."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    isz = {'b': 1, 'B': 1, 'h': 2, 'i': 4, 'f': 4, 'd': 8}[enc]
    n = 3 * (CB // (2 * isz))
    body = signals.generic_bytes(enc, n, 17 + q, 1_000_000, center or 40_000, big_endian=False)
    kw = dict(fs=1_000_000, enc=enc, center=center, dec=q, demod=demod, omega_out=4000, correct_iq=iq,
              vfos=None, simo=False, normalize=norm, swap=False, big_endian=None)
    pl = plan_for(kw)
    with Engine(pl, max_chunks=3, keep_decimated=True) as eng:
        assert eng.tc is None                                   # none of these shapes is a GEMM shape
        out = eng.process(body)
        off = eng.iq_state
    ch = orc.Chain(**kw)
    ref = ch.run(body)
    assert out.shape == ref.shape and rel_err(out, ref) < TOL
    if iq:
        assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))


def _sweep_cases():
    """A fixed pseudo-random sweep over what the CLI accepts: encoding x byte order x decimation x
    demodulation x --correct-iq x --normalize-input x centre, single VFO and small banks."""
    rng = np.random.default_rng(20261018)
    qs = [6, 7, 9, 12, 20, 31, 33, 48, 100, 127, 130, 200, 256]
    out = []
    for i in range(16):
        enc = 'bBhHiIfd'[i % 8]
        q = int(qs[int(rng.integers(len(qs)))])
        demod = ['fm', 'am', 're', 'im'][int(rng.integers(4))]
        if demod == 'fm' and q < 8:
            demod = 'am'
        iq = bool(rng.integers(2))
        norm = bool(rng.integers(2)) and enc in 'bBhHiI'
        swap = bool(rng.integers(2)) and enc not in 'bB'
        center = int(rng.integers(-200, 200)) * 1000
        simo = i % 5 == 4
        out.append((enc, q, demod, iq, norm, swap, center, simo))
    return out


@pytest.mark.parametrize('enc,q,demod,iq,norm,swap,center,simo', _sweep_cases())
def test_option_sweep_against_the_oracle(enc, q, demod, iq, norm, swap, center, simo):
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    isz = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'i': 4, 'I': 4, 'f': 4, 'd': 8}[enc]
    n = 2 * (CB // (2 * isz))
    body = signals.generic_bytes(enc, n, 100 + q, 1_000_000, center or 40_000, big_endian=swap)
    kw = dict(fs=1_000_000, enc=enc, center=0 if simo else center, dec=q, demod=demod, omega_out=min(4000, 1_000_000 // q // 5), correct_iq=iq,
              vfos='-30000,25000,110000' if simo else None, simo=simo, normalize=norm, swap=swap, big_endian=None)
    pl = plan_for(kw)
    with Engine(pl, max_chunks=2) as eng:
        out = eng.process(body)
        off = eng.iq_state
    ch = orc.Chain(**kw)
    ref = ch.run(body)
    got = np.asarray(out, dtype=np.float64)
    assert got.shape == ref.shape
    for r in range(pl.R):
        assert rel_err(got[r], ref[r]) < TOL, (r, rel_err(got[r], ref[r]))
    if iq:
        assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))


@pytest.mark.parametrize('enc,q,demod', [('H', 256, 'fm'), ('I', 128, 'im'), ('i', 256, 'am'), ('d', 128, 'fm'), ('h', 128, 'fm')])
def test_fused_finish_kernel_on_short_rows(enc, q, demod):
    """k_finish with rows of 64 / 128 / 256 outputs per chunk (4-byte and wider samples at large
    -d): its phase-1 scratch overlays the FFT buffer and the output row, and for rows of 128 and
    fewer the scratch is the larger of the two (the per-warp region was sized for the row only:
    neighbouring warps raced).  Many chunks, so that all warps of a CTA are busy."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    isz = {'h': 2, 'H': 2, 'i': 4, 'I': 4, 'd': 8}[enc]
    nch = 24
    n = nch * (CB // (2 * isz))
    body = signals.generic_bytes(enc, n, 7 + q, 1_000_000, 30_000, big_endian=False)
    kw = dict(fs=1_000_000, enc=enc, center=30000, dec=q, demod=demod, omega_out=min(4000, 1_000_000 // q // 5), correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=False, big_endian=None)
    pl = plan_for(kw)
    assert pl.M in (64, 128, 256) and pl.rem == 0
    with Engine(pl, max_chunks=nch) as eng:
        out = eng.process(body)
    ref = orc.Chain(**kw).run(body)
    assert out.shape == ref.shape and rel_err(out, ref) < TOL


def _tc_sweep_cases():
    """The shapes the tensor-core front end takes (8-bit at -d 64 / 128, 16-bit at -d 32 / 64),
    crossed with byte order, demodulation, --correct-iq, centre and bank width."""
    rng = np.random.default_rng(7)
    shapes = [('b', 64), ('b', 128), ('B', 64), ('B', 128), ('h', 32), ('h', 64), ('H', 32), ('H', 64)]
    out = []
    for i in range(12):
        enc, q = shapes[i % 8]
        demod = ['fm', 'am', 're', 'im'][int(rng.integers(4))]
        iq = bool(rng.integers(2))
        swap = bool(rng.integers(2)) and enc in 'hH'
        center = int(rng.integers(-300, 300)) * 1000
        nv = [0, 0, 2, 7, 31][int(rng.integers(5))]
        out.append((enc, q, demod, iq, swap, center, nv))
    return out


@pytest.mark.parametrize('enc,q,demod,iq,swap,center,nv', _tc_sweep_cases())
def test_tensor_core_option_sweep_against_the_oracle(enc, q, demod, iq, swap, center, nv):
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    isz = 1 if enc in 'bB' else 2
    nch = 3
    n = nch * (CB // (2 * isz))
    vfos = ','.join(str(int(v)) for v in np.linspace(-400_000, 400_000, nv)) if nv else None
    if nv and demod == 'fm':
        # the phase of a row without a carrier is ill-conditioned (|d phi| = |dy| / |y| with y the
        # stop-band residue): give every row of the bank its own carrier
        rng = np.random.default_rng(300 + q + nv)
        kind, lo, hi, amp, dc = {'b': ('i1', -128, 127, 3.5, 0.0), 'B': ('u1', 0, 255, 3.5, 127.5),
                                 'h': ('i2', -32768, 32767, 900.0, 0.0), 'H': ('u2', 0, 65535, 900.0, 32768.0)}[enc]
        z = np.full(n, dc * (1 + 1j), dtype=np.complex128)
        for i, f in enumerate([int(v) for v in np.linspace(-400_000, 400_000, nv)] + [0]):
            z += signals._fm_carrier(n, 1_000_000, f, 600 + 25 * i, 1_500, amp, phase0=0.2 * i)
        z = z + amp * 0.05 * (rng.normal(0, 1, n) + 1j * rng.normal(0, 1, n))
        body = signals._interleave(z, np.dtype(kind).newbyteorder('>' if swap else '<'), lo, hi).tobytes()
    else:
        body = signals.generic_bytes(enc, n, 300 + q + nv, 1_000_000, center or 40_000, big_endian=swap)
    kw = dict(fs=1_000_000, enc=enc, center=0 if nv else center, dec=q, demod=demod, omega_out=3000, correct_iq=iq,
              vfos=vfos, simo=bool(nv), normalize=False, swap=swap, big_endian=None)
    pl = plan_for(kw)
    with Engine(pl, max_chunks=nch) as eng:
        assert eng.tc is not None and pl.R == (nv + 1 if nv else 1)
        out = eng.process(body)
        off = eng.iq_state
    ch = orc.Chain(**kw)
    ref = ch.run(body)
    got = np.asarray(out, dtype=np.float64)
    assert got.shape == ref.shape
    for r in range(pl.R):
        assert rel_err(got[r], ref[r]) < TOL, (r, rel_err(got[r], ref[r]))
    if iq:
        assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))
