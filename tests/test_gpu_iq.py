"""GPU: the complex baseband output (``-m iq``) against its oracle (tests/iq_ref.py), bit-exact
against separate ``-m re`` / ``-m im`` runs, through every layer: the fused k_finish, the general
k_fixup + k_demod path, the seamless mode, the banks, submit/wait, the operator, the CLI and the
multi-GPU drivers in a one-rank group."""
import os

import numpy as np
import pytest

import signals
from gpu_util import chunked
from iq_ref import iq_oracle, seamless_iq_oracle
from oracle import oracle as orc
from sdrterm_b200.plan import build_plan
from util import parse_wav, rel_err

TOL = 1e-9
_ISZ = {'b': 1, 'B': 1, 'h': 2, 'H': 2, 'f': 4, 'd': 8}


def _kw(enc, q, iq, center, fs=1_024_000, norm=False, swap=False, simo=False, vfos=None, demod='iq'):
    return dict(fs=fs, enc=enc, center=center, dec=q, demod=demod, omega_out=5000, correct_iq=iq, vfos=vfos,
                simo=simo, normalize=norm, swap=swap, big_endian=None)


def _plan(kw, seamless=False):
    ch = orc.Chain(**{**kw, 'demod': 're'})
    return build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, simo=kw['simo'], swap=orc.needs_swap(ch.dt),
                      correct_iq=kw['correct_iq'], normalize=kw['normalize'], demod=kw['demod'],
                      omega_out=kw['omega_out'], seamless=seamless)


def _body(kw, nch, seed, extra=0):
    n = nch * 131072 // (2 * _ISZ[kw['enc']]) + extra
    return signals.generic_bytes(kw['enc'], n, seed, kw['fs'], kw['center'] or 40_000, big_endian=kw['swap'])


def _process(kw, body, use_tc=True, max_chunks=8):
    from sdrterm_b200.engine import Engine
    pl = _plan(kw)
    with Engine(pl, max_chunks=max_chunks, use_tc=use_tc) as eng:
        assert eng.W == pl.W == (2 * pl.M if kw['demod'] == 'iq' else pl.M)
        tc = eng.tc is not None
        out = np.asarray(eng.process(chunked(body)), dtype=np.float64)
    return out, pl, tc


# name, kw, use_tc, expected front end (True = k_tc)
CASES = [
    ('b d64 iq c20k', _kw('b', 64, True, 20000, fs=250_000), True, True),
    ('b-swap d64', _kw('b', 64, False, 20000, fs=250_000, swap=True), True, True),
    ('B d64 norm c0', _kw('B', 64, True, 0, fs=2_400_000, norm=True), True, False),
    ('B-swap d64 iq', _kw('B', 64, True, -30000, fs=2_400_000, swap=True), True, True),
    ('h d64 iq k_tc', _kw('h', 64, True, 15000), True, True),
    ('h d64 iq k_main', _kw('h', 64, True, 15000), False, False),
    ('h-swap d32 c0', _kw('h', 32, False, 0, swap=True), True, True),
    ('H d32 norm iq', _kw('H', 32, True, -50000, fs=1_000_000, norm=True), True, False),
    ('H-swap d32 iq', _kw('H', 32, True, -50000, fs=1_000_000, swap=True), True, True),
    ('f d256 c30k', _kw('f', 256, False, 30000, fs=2_400_000), True, False),
    ('f-swap d64 iq', _kw('f', 64, True, 30000, fs=2_400_000, swap=True), True, False),
    ('d d32 iq', _kw('d', 32, True, 12000, fs=192_000), True, False),
    ('d-swap d4 norm c0', _kw('d', 4, False, 0, fs=192_000, swap=True, norm=True), True, False),
    ('h d50 ragged iq', _kw('h', 50, True, 15000), True, False),
    ('B d25 odd iq', _kw('B', 25, True, 10000, fs=2_400_000), True, False),
    ('h d5 odd norm', _kw('h', 5, False, 30000, norm=True), True, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,kw,use_tc,want_tc', CASES, ids=[c[0] for c in CASES])
def test_iq_matches_oracle(name, kw, use_tc, want_tc):
    body = _body(kw, 2, 300 + kw['dec'], extra=1000)       # 3 chunks, the last one with a stale tail
    out, pl, tc = _process(kw, body, use_tc)
    assert tc == want_tc
    ref = iq_oracle(kw, body)
    err = rel_err(out, ref)
    print(f'{name}: M={pl.M} err={err:.3e}')
    assert out.shape == ref.shape == (1, 3 * 2 * pl.M) and err < TOL


def _re_im_iq(kw, body, use_tc=True):
    outs = {}
    for demod in ('re', 'im', 'iq'):
        outs[demod], pl, _ = _process({**kw, 'demod': demod}, body, use_tc)
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize('kw,general', [
    (_kw('h', 64, True, 15000), False),                            # fused k_finish (k_tc)
    (_kw('B', 64, True, 0, fs=2_400_000, norm=True), False),       # fused k_finish (k_main)
    (_kw('h', 64, True, 15000), True),                             # general path forced
    (_kw('h', 50, True, 15000), True),                             # general path: ragged blocks
    (_kw('B', 25, False, -20000, fs=2_400_000), True),             # general path: odd -d
], ids=['fused-tc', 'fused-main', 'general-forced', 'general-d50', 'general-d25'])
def test_iq_columns_are_bit_identical_to_re_and_im(kw, general, monkeypatch):
    if general:
        monkeypatch.setenv('SDRB_NO_FINISH', '1')
    body = _body(kw, 3, 21)
    o = _re_im_iq(kw, body)
    assert np.array_equal(o['iq'][:, 0::2], o['re'])
    assert np.array_equal(o['iq'][:, 1::2], o['im'])


@pytest.mark.gpu
def test_iq_banks_match_oracle():
    """Config 3's 17-row big-endian SIMO bank (k_tc) and config 4's 257-row float32 bank (k_main)."""
    from sdrterm_b200.engine import Engine
    body, vfos = signals.c3_bytes(2 * 32768, seed=3)
    kw = _kw('h', 64, False, 0, fs=2_400_000, swap=True, simo=True, vfos=vfos)
    pl = _plan(kw)
    assert pl.R == 17 and pl.big_endian_out
    with Engine(pl, max_chunks=2) as eng:
        raw = eng.process(chunked(body))
        assert eng.tc is not None
    assert raw.dtype == np.dtype('>f8')
    ref = iq_oracle(kw, body)
    assert raw.shape == ref.shape and rel_err(np.asarray(raw, dtype=np.float64), ref) < TOL
    body4, vfos4 = signals.c4_bytes(2 * 16384, seed=4)
    kw4 = _kw('f', 64, False, 0, fs=61_440_000, simo=True, vfos=vfos4)
    pl4 = _plan(kw4)
    assert pl4.R == 257
    with Engine(pl4, max_chunks=2) as eng:
        out4 = np.asarray(eng.process(chunked(body4)), dtype=np.float64)
        assert eng.tc is None
    ref4 = iq_oracle(kw4, body4)
    assert out4.shape == ref4.shape and rel_err(out4, ref4) < TOL


@pytest.mark.gpu
def test_iq_submit_wait_alternating_slots():
    from sdrterm_b200._native import PinnedBuffer
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, True, 15000)
    pl = _plan(kw)
    sizes = [1, 3, 2, 4, 1, 2, 3]
    body = _body(kw, sum(sizes), 5)
    cb = pl.chunk_bytes
    with Engine(pl, max_chunks=4) as eng:
        hin = [PinnedBuffer(4 * cb) for _ in range(2)]
        hout = [PinnedBuffer(eng.R * 4 * eng.W * 8) for _ in range(2)]
        parts, pending, o = [], [0, 0], 0

        def collect(s):
            eng.wait(s)
            parts.append(hout[s].view(np.float64)[:eng.W * pending[s]].copy())
            pending[s] = 0

        for b, n in enumerate(sizes):          # batch b on slot b & 1 while batch b - 1 is in flight
            s = b & 1
            if pending[s]:
                collect(s)                     # batch b - 2
            hin[s].u8[:n * cb] = np.frombuffer(body[o:o + n * cb], dtype=np.uint8)
            eng.submit(s, hin[s].ptr.value, n, hout[s].ptr.value)
            pending[s] = n
            o += n * cb
        collect(len(sizes) & 1)
        collect((len(sizes) - 1) & 1)
    out = np.concatenate(parts)[None]
    ref = iq_oracle(kw, body)
    assert out.shape == ref.shape and rel_err(out, ref) < TOL


def _stream(eng, body, splits):
    cb = eng.chunk_bytes
    outs, o, i, counts = [], 0, 0, []
    while o < len(body):
        k = splits[i % len(splits)]
        i += 1
        r = eng.stream(body[o:o + k * cb])
        assert r.shape[1] % eng.W == 0
        counts.append(r.shape[1] // eng.W)
        outs.append(np.asarray(r, dtype=np.float64))
        o += k * cb
    outs.append(np.asarray(eng.stream_end(), dtype=np.float64))
    return np.concatenate(outs, axis=1), counts


@pytest.mark.gpu
@pytest.mark.parametrize('kw', [_kw('h', 64, True, 15000), _kw('f', 256, True, 30000, fs=2_400_000)],
                         ids=['int16-d64', 'float32-d256'])
def test_seamless_iq_matches_oracle_across_batch_splits(kw):
    from sdrterm_b200.engine import Engine
    pl = _plan(kw, seamless=True)
    D = pl.lookahead
    nch = 3 * (D + 1) + 2
    body = _body(kw, nch, 11)
    ref, _ = seamless_iq_oracle(kw, body)
    res = []
    with Engine(pl, max_chunks=8) as eng:
        assert eng.lookahead == D and eng.W == 2 * pl.M
        for split in (1, 2, 5, 8):
            out, counts = _stream(eng, body, (split,))
            seen, emitted = 0, 0
            for k in counts:                       # per call: max(0, seen - D) - emitted chunks
                seen = min(nch, seen + split)
                assert k == max(0, seen - D) - emitted
                emitted += k
            assert out.shape[1] == nch * pl.W     # stream_end emitted the rest
            res.append(out)
    for o in res[1:]:
        assert rel_err(o, res[0]) <= 1e-12
    err = rel_err(res[0], ref)
    print(f'seamless iq D={D}: err={err:.3e}')
    assert res[0].shape == ref.shape and err < TOL


@pytest.mark.gpu
def test_seamless_iq_bank_and_exactness():
    """The 17-row big-endian bank in seamless mode against the oracle, and the seamless iq columns
    bit-identical to seamless re / im runs."""
    from sdrterm_b200.engine import Engine
    body, vfos = signals.c3_bytes(4 * 32768, seed=3)
    kw = _kw('h', 64, False, 0, fs=2_400_000, swap=True, simo=True, vfos=vfos)
    outs = {}
    for demod in ('re', 'im', 'iq'):
        pl = _plan({**kw, 'demod': demod}, seamless=True)
        with Engine(pl, max_chunks=4) as eng:
            outs[demod], _ = _stream(eng, body, (3, 1))
    ref, _ = seamless_iq_oracle(kw, body)
    assert outs['iq'].shape == ref.shape and rel_err(outs['iq'], ref) < TOL
    assert np.array_equal(outs['iq'][:, 0::2], outs['re'])
    assert np.array_equal(outs['iq'][:, 1::2], outs['im'])


@pytest.mark.gpu
@pytest.mark.parametrize('M', [512, 1311])
def test_iq_operator_matches_real_and_imag(M):
    from sdrterm_b200.dsp import demodulation as dem
    rng = np.random.default_rng(M)
    y = rng.normal(size=(3, M)) + 1j * rng.normal(size=(3, M))
    res = np.empty((3, 2 * M))
    re_, im_ = np.empty((3, M)), np.empty((3, M))
    dem.iqOutput(y, res)
    dem.realOutput(y, re_)
    dem.imagOutput(y, im_)
    assert np.array_equal(res[:, 0::2], re_) and np.array_equal(res[:, 1::2], im_)
    assert np.array_equal(res.view(np.complex128), y)


@pytest.mark.gpu
def test_iq_refuses_smoothing():
    from sdrterm_b200 import _native as nat
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    from sdrterm_b200.engine import Engine
    pl = _plan(_kw('h', 64, True, 15000))
    with pytest.raises(ValueError):
        Engine(pl, max_chunks=1, smooth=5)
    with Engine(pl, max_chunks=1) as eng:
        with pytest.raises(ValueError):
            eng.set_smooth(5)
        rc = nat.lib().sdrb_set_smooth(eng._h, 5, 2, 2, -2, np.zeros(25).ctypes.data)
        assert rc == -1
        assert nat.lib().sdrb_set_smooth(eng._h, 0, 0, 0, 0, None) == 0        # switching off stays allowed
    p = DspProcessor(1_024_000, center=15000, dec=64, enc='h', smooth=5)
    p.selectOutputIq()
    with pytest.raises(ValueError):
        p._makeEngine(b'\0' * 131072)


def _cli_env():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return dict(os.environ, PYTHONPATH=os.path.join(root, 'src'))


@pytest.mark.gpu
def test_cli_iq_wav_equals_engine(tmp_path):
    import subprocess
    import sys
    from sdrterm_b200.engine import Engine
    raw = signals.c1_bytes(3 * 32768 + 5000, seed=0)
    fin, fout = tmp_path / 'in.wav', tmp_path / 'out.bin'
    fin.write_bytes(raw)
    subprocess.run([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-o', str(fout), '-c', '15000',
                    '-d', '64', '-m', 'iq', '--correct-iq'], env=_cli_env(), cwd=str(tmp_path),
                   check=True, timeout=300, capture_output=True)
    fs, enc, be, off = parse_wav(raw)
    kw = _kw(enc, 64, True, 15000, fs=fs)
    with Engine(_plan(kw), max_chunks=8) as eng:
        want = eng.process(chunked(raw[off:]))
    got = np.frombuffer(fout.read_bytes(), dtype='=f8')[None]
    assert got.shape == want.shape == (1, 4 * 2 * 512)
    assert rel_err(got, want) < 1e-13                       # batches may split differently (IQ state chain)
    assert rel_err(got, iq_oracle(kw, raw[off:])) < TOL


@pytest.mark.gpu
def test_cli_simo_iq_sockets(tmp_path):
    """`--simo -m iq`: every VFO socket receives 2M big-endian doubles per chunk, its row of the oracle."""
    import socket
    import subprocess
    import sys
    import threading
    import time
    nch = 3
    body, vfos = signals.c3_bytes(nch * 32768, seed=3)
    vf = ','.join(vfos.split(',')[:2])
    fin = tmp_path / 'in.raw'
    fin.write_bytes(body)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    proc = subprocess.Popen([sys.executable, '-m', 'sdrterm', '-i', str(fin), '-r', '2400k', '-e', 'h', '-X', '-d', '64',
                             '-m', 'iq', '--simo', f'--vfos={vf}', '--vfo-host', f'127.0.0.1:{port}'],
                            env=_cli_env(), cwd=str(tmp_path), stderr=subprocess.PIPE, text=True)
    head = ''
    deadline = time.time() + 120
    while time.time() < deadline and 'Accepting' not in head:
        line = proc.stderr.readline()
        if not line:
            break
        head += line
    got = {}

    def client(i):
        c = socket.create_connection(('127.0.0.1', port), timeout=30)
        buf = b''
        while True:
            d = c.recv(1 << 16)
            if not d:
                break
            buf += d
        got[i] = buf
        c.close()

    cl = [threading.Thread(target=client, args=(i,), daemon=True) for i in range(3)]
    for t in cl:
        t.start()
    proc.stderr.read()
    proc.wait(120)
    for t in cl:
        t.join(30)
    kw = _kw('h', 64, False, 0, fs=2_400_000, swap=True, simo=True, vfos=vf)
    ref = iq_oracle(kw, body)
    M = 32768 // 64
    assert sorted(got) == [0, 1, 2]
    for i in range(3):
        assert len(got[i]) == nch * 2 * M * 8
        g = np.frombuffer(got[i], dtype='>f8').astype(np.float64)
        assert min(rel_err(g, r) for r in ref) < TOL


@pytest.mark.gpu
def test_multigpu_drivers_carry_iq_rows_in_a_one_rank_group(tmp_path):
    import torch
    import torch.distributed as dist
    from sdrterm_b200 import multigpu
    from sdrterm_b200.engine import Engine
    kw = _kw('h', 64, True, 15000)
    pl = _plan(kw)
    nch = 3
    body = signals.c1_bytes(nch * 32768, seed=9, header=False)
    with Engine(pl, max_chunks=nch) as eng:
        want = np.asarray(eng.process(body), dtype=np.float64)
    dist.init_process_group('gloo', init_method=f'file://{tmp_path}/pg', rank=0, world_size=1)
    try:
        dev = torch.device('cuda', 0)
        raw = torch.from_numpy(np.frombuffer(body, dtype=np.uint8).copy()).to(dev)
        chain = multigpu.TimeShardedChain(pl, max_chunks=nch, device=0, dist=dist, torch=torch)
        out = torch.empty((1, nch * pl.W), dtype=torch.float64, device=dev)
        chain.step(raw.data_ptr(), nch, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        chain.close()
        assert np.array_equal(out.cpu().numpy(), want)
        path = tmp_path / 'in.raw'
        path.write_bytes(body)
        got = multigpu.run_file_sharded(str(path), None, fs=1_024_000, enc='h', dec=64, center=15000, demod='iq',
                                        correct_iq=True, batch_chunks=2, device=0, dist=dist, torch=torch)
        assert got.shape == want.shape and rel_err(got, want) < 1e-13       # batches of 2 + 1 chunks
        bvfos = [100_000, -200_000]
        bank = multigpu.RowShardedBank(2_400_000, 'h', 64, bvfos + [0], max_chunks=nch, device=0, dist=dist, torch=torch,
                                       demod='iq', omega_out=5000)
        assert bank.W == 2 * bank.M
        outs = [torch.empty((3, nch * bank.W), dtype=torch.float64, device=dev)]
        bank.run([raw], nch, outs, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        bank.close()
        bkw = _kw('h', 64, False, 0, fs=2_400_000, simo=True, vfos=','.join(str(v) for v in bvfos))
        bref = iq_oracle(bkw, body)
        bgot = outs[0].cpu().numpy().view('>f8').astype(np.float64)
        assert bgot.shape == bref.shape and rel_err(bgot, bref) < TOL
    finally:
        dist.destroy_process_group()
