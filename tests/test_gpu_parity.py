"""GPU parity: the CUDA path through the C ABI vs the oracle, vs the numpy emulator of the
kernels, and vs the reference's golden outputs.  Tolerance from BASELINE.json's north_star:
max|out - ref| / max|ref| <= 1e-9 on the float64 output (observed ~1e-12); integer decode and
output sample counts exact."""
import numpy as np
import pytest

from cases import CASES
from oracle import oracle as orc
from util import case_stream, load_golden, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _tc_ok(name):
    from gpu_util import plan_for
    from sdrterm_b200.plan import tc_supported
    from util import case_stream as cs
    return tc_supported(plan_for(cs(name)[2]))


@pytest.mark.parametrize('path', ['fp64', 'tc'])
@pytest.mark.parametrize('name', sorted(CASES))
def test_case_vs_oracle_and_golden(name, path):
    """Both block front ends: 'fp64' = k_main (FP64 tensor pipe, any shape), 'tc' = k_tc (tcgen05
    int8 GEMM over the raw bytes, 8/16-bit integer encodings with 128- or 256-byte blocks)."""
    from gpu_util import run_case
    if path == 'tc' and not _tc_ok(name):
        pytest.skip('shape not handled by the tensor-core front end (falls back to k_main)')
    kw, pl, chunks, out, y, off = run_case(name, use_tc=(path == 'tc'))
    g = load_golden(name)
    ch = orc.Chain(**kw)
    zs = np.stack([ch.ingest(c.tobytes()).copy() for c in chunks])
    yo = ch.decimated(zs)
    oo = np.concatenate([ch.demodulate(yo[c]) for c in range(len(chunks))], axis=1)
    got = np.asarray(out, dtype=np.float64)          # undoes big-endian framing
    assert got.shape == oo.shape == g['out'].shape   # sample count / indexing exact
    assert rel_err(y, yo) < TOL
    assert rel_err(got, oo) < TOL
    assert rel_err(got, g['out']) < TOL
    assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))
    if pl.big_endian_out:
        assert out.dtype == np.dtype('>f8')


@pytest.mark.parametrize('name', ['c1_fm_wav_int16', 'c2_am_u8_d50_ceil', 'c3_simo16_int16be'])
def test_stage_parity_vs_emulator(name):
    """Decimator output chunk by chunk vs tests/emulator.py (same tables, same algorithm)."""
    import emulator as emu
    from gpu_util import run_case
    from sdrterm_b200.plan import build_tc
    kw, pl, chunks, out, y, off = run_case(name)
    tc = build_tc(pl)
    if tc is not None:      # the tensor-core front end ran: its own twin (same digit matrices)
        eo, ey, eoff = emu.emu_stream_tc(pl, tc, chunks.tobytes())
    else:
        eo, ey, eoff = emu.emu_stream(pl, chunks.tobytes())
    assert rel_err(y, ey) < 1e-11
    assert rel_err(np.asarray(out, dtype=np.float64), eo) < 1e-11
    if tc is not None:      # and the FP64 block kernel against the general twin
        kw, pl, chunks, out2, y2, off2 = run_case(name, use_tc=False)
        eo2, ey2, _ = emu.emu_stream(pl, chunks.tobytes())
        assert rel_err(y2, ey2) < 1e-11


@pytest.mark.parametrize('name', ['c1_fm_wav_int16', 'c2_am_u8_d64', 'c3_simo16_int16be', 'enc_H_swap_im'])
def test_general_finish_kernels_match_fused(name, monkeypatch):
    """k_fixup + k_demod (the general path, forced with SDRB_NO_FINISH=1) against the fused
    k_finish on shapes both handle, and against the oracle.  Both paths take the chunk gains and the
    chunk scan from the same kernels, so the IQ state is bit-identical."""
    from gpu_util import run_case
    kw, pl, chunks, out_f, y_f, off_f = run_case(name)
    monkeypatch.setenv('SDRB_NO_FINISH', '1')
    kw, pl, chunks, out_g, y_g, off_g = run_case(name)
    ch = orc.Chain(**kw)
    oo = ch.run(chunks.tobytes())
    assert rel_err(y_g, y_f) < 1e-12
    assert rel_err(np.asarray(out_g, dtype=np.float64), np.asarray(out_f, dtype=np.float64)) < 1e-11
    assert rel_err(np.asarray(out_g, dtype=np.float64), oo) < TOL
    assert off_g == off_f


def test_batch_split_and_state_carry():
    """Feeding chunk by chunk (max_chunks=1) equals one batch: the IQ state chains.  The same on
    the general IQ path (k_iqgain -> k_iqscan_c -> k_iqtiles) with 9000 small ragged chunks in one
    batch, more than the 8192 that k_iqscan_c scans per round: against the oracle, offset included,
    and against batches of 1000."""
    import signals
    from gpu_util import chunked, plan_for
    from sdrterm_b200.engine import Engine
    from sdrterm_b200.plan import build_plan
    raw, body, kw = case_stream('c1_fm_wav_int16')
    pl = plan_for(kw)
    chunks = chunked(body)
    with Engine(pl, max_chunks=8) as e1:
        a = e1.process(chunks)
    with Engine(pl, max_chunks=1) as e2:
        b = np.concatenate([e2.process(chunks[c]) for c in range(len(chunks))], axis=1)
    with Engine(pl, max_chunks=2) as e3:
        c = e3.process(chunks)            # internal batching path
    assert rel_err(b, a) < 1e-13 and rel_err(c, a) < 1e-13

    nch, cb = 9000, 1024                  # 256 samples per chunk at -d 50: 5 blocks + 6 samples
    body = signals.c1_bytes(nch * cb // 4, seed=13, header=False)
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=50, demod='am', omega_out=5000, correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=False, big_endian=None, chunk_bytes=cb)
    ch = orc.Chain(**kw)
    pl = build_plan(kw['fs'], 'h', 50, ch.rows, correct_iq=True, demod='am', omega_out=5000, chunk_bytes=cb)
    assert pl.rem != 0
    with Engine(pl, max_chunks=nch) as e4:
        whole = e4.process(body)
        off = e4.iq_state
    with Engine(pl, max_chunks=1000) as e5:
        split = e5.process(body)
    ref = ch.run(body)
    assert whole.shape == ref.shape and rel_err(whole, ref) < TOL
    assert abs(off - ch._off[0]) <= 1e-9 * max(1.0, abs(ch._off[0]))
    assert rel_err(split, whole) < 1e-13


def test_tc_long_stream_matches_oracle_and_fp64_path():
    """Many MMA tiles per CTA (persistent loop, both accumulator stages, barrier phases wrap):
    300 chunks of the config-1 stream through k_tc vs the oracle and vs the FP64 block kernel."""
    import signals
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    nch = 300
    base = signals.c1_bytes(20 * 32768, seed=7, header=False)
    body = (base * (nch // 20))[:nch * 131072]
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=False, big_endian=None)
    pl = plan_for(kw)
    with Engine(pl, max_chunks=nch, use_tc=True, keep_decimated=True) as e1:
        assert e1.tc is not None
        a = e1.process(body)
        ya = e1.decimated(nch)
        offa = e1.iq_state
    with Engine(pl, max_chunks=nch, use_tc=False, keep_decimated=True) as e2:
        b = e2.process(body)
        yb = e2.decimated(nch)
        offb = e2.iq_state
    ref = orc.Chain(**kw, nthreads=orc.max_threads()).run_fast(body)
    assert a.shape == b.shape == ref.shape
    assert rel_err(ya, yb) < 1e-11
    assert rel_err(a, ref) < TOL and rel_err(b, ref) < TOL
    assert abs(offa - offb) <= 1e-9 * max(1.0, abs(offb))


def test_time_segment_phases_with_device_side_iq_exchange():
    """Two 'ranks' on one GPU: each runs MAIN|IQSCAN from a zero offset, exports its gain, the gains
    are folded on the device (sdrb_iq_prefix_device) and IQSCAN|FINISH completes; the concatenation
    equals one pass over the whole stream (SURVEY 8e, config 5)."""
    import torch
    import signals
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True,
              vfos=None, simo=False, normalize=False, swap=False, big_endian=None)
    pl = plan_for(kw)
    body = np.frombuffer(signals.c1_bytes(12 * 32768, seed=9, header=False), dtype=np.uint8)
    segs = [(0, 7), (7, 5)]
    with Engine(pl, max_chunks=12) as e0:
        whole = e0.process(body)
    raw = torch.from_numpy(body.copy()).cuda()
    gains = torch.zeros(6, dtype=torch.float64, device='cuda')
    outs, engs = [], []
    for r, (s, n) in enumerate(segs):
        e = Engine(pl, max_chunks=n)
        engs.append(e)
        e.process_device_phases(raw.data_ptr() + s * 131072, n, 0, 1 | 2 | 8)
        e.iq_export_device(gains.data_ptr() + 24 * r, n * 32768)
    for r, (s, n) in enumerate(segs):
        o = torch.empty((1, n * pl.M), dtype=torch.float64, device='cuda')
        engs[r].iq_prefix_device(gains.data_ptr(), r)
        engs[r].process_device_phases(raw.data_ptr() + s * 131072, n, o.data_ptr(), 2 | 4)
        outs.append(o)
    torch.cuda.synchronize()
    got = torch.cat(outs, dim=1).cpu().numpy()
    for e in engs:
        e.close()
    assert got.shape == whole.shape and rel_err(got, whole) < 1e-12


def test_empty_and_single_chunk_batches():
    """Edge sizes: no chunks at all, and one chunk (fewer MMA tiles than SMs) on the tensor-core path."""
    from gpu_util import plan_for
    from sdrterm_b200.engine import Engine
    raw, body, kw = case_stream('c1_fm_wav_int16')
    pl = plan_for(kw)
    with Engine(pl, max_chunks=4) as e:
        out0 = e.process(b'')
        assert out0.shape == (1, 0)
        one = e.process(body[:131072])
        with pytest.raises(ValueError):
            e.process(body[:131072 + 5])              # not a whole number of chunks
    ref = orc.Chain(**kw).run(body[:131072])
    assert one.shape == ref.shape and rel_err(one, ref) < TOL


def test_full_size_linearity_and_batch_invariance():
    """BASELINE-size batch (8192 chunks = 2^28 samples, 1 GiB of int16 IQ) through size-independent
    properties: the chain up to the decimator is linear (re output, IQ correction on), so
    out(a) + out(b) == out(a + b); and one 8192-chunk call equals eight 1024-chunk calls (the IQ
    state chains).  Device-resident buffers, C ABI entry point sdrb_process_device."""
    import torch
    from sdrterm_b200.engine import Engine
    from sdrterm_b200.plan import build_plan
    nch = 8192
    pl = build_plan(1_024_000, 'h', 64, [15000], correct_iq=True, demod='re', omega_out=5000)
    g = torch.Generator(device='cuda')
    g.manual_seed(11)
    n = nch * 32768 * 2
    a = torch.randint(-12000, 12000, (n,), generator=g, device='cuda', dtype=torch.int16)
    b = torch.randint(-12000, 12000, (n,), generator=g, device='cuda', dtype=torch.int16)
    c = a + b
    outs = []
    with Engine(pl, max_chunks=nch) as e:
        assert e.tc is not None
        for x in (a, b, c):
            o = torch.empty((1, nch * pl.M), dtype=torch.float64, device='cuda')
            e.iq_state = 0j
            e.process_device(x.data_ptr(), nch, o.data_ptr())
            torch.cuda.synchronize()
            outs.append(o)
        ssum = outs[0] + outs[1]
        err = float((ssum - outs[2]).abs().max() / outs[2].abs().max())
        assert err < 1e-11, err
        # eight batches of 1024 chunks with the state carried == one batch
        o8 = torch.empty_like(outs[2])
        e.iq_state = 0j
        for k in range(8):
            tmp = torch.empty((1, 1024 * pl.M), dtype=torch.float64, device='cuda')
            e.process_device(c.data_ptr() + k * 1024 * 131072, 1024, tmp.data_ptr())
            torch.cuda.synchronize()
            o8[0, k * 1024 * pl.M:(k + 1) * 1024 * pl.M] = tmp[0]
        err8 = float((o8 - outs[2]).abs().max() / outs[2].abs().max())
        assert err8 < 1e-12, err8
    # spot check of the first and last chunk against the oracle
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='re', omega_out=5000, correct_iq=True)
    host = c[:32768 * 2].cpu().numpy().tobytes()
    ref0 = orc.Chain(**kw).run(host)
    assert rel_err(outs[2][0, :pl.M].cpu().numpy()[None], ref0) < TOL
