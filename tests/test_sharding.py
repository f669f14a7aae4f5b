"""Multi-process (world size 2, gloo, CPU) coverage of the N>1 paths: time-segment sharding with
the IQ-offset hand-off, and VFO-row sharding with the raw-chunk broadcast.  The compute engine in
these CPU tests is the oracle (the checker); what is under test is sdrterm_b200/sharding.py."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from sdrterm_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CB = 131072


def test_partitions_cover_everything_once():
    for n in (1, 2, 7, 17, 257):
        for w in (1, 2, 3, 4, 8):
            rows = [sharding.row_shard(n, w, r) for r in range(w)]
            assert rows[0][0] == 0 and rows[-1][1] == n
            assert all(rows[i][1] == rows[i + 1][0] for i in range(w - 1))
            cnt = [b - a for a, b in rows]
            assert max(cnt) - min(cnt) <= 1 and cnt == sorted(cnt, reverse=True)
            segs = [sharding.segment_shard(n, w, r) for r in range(w)]
            assert sum(c for _, c in segs) == n
            assert all(segs[i][0] + segs[i][1] == segs[i + 1][0] for i in range(w - 1))
            assert max(c for _, c in segs) - min(c for _, c in segs) <= 1


def test_iq_prefix_equals_serial_recurrence():
    rng = np.random.default_rng(0)
    lam, L = 1 - 50 / 1_024_000, 50 / 1_024_000
    z = rng.normal(size=3000) + 1j * rng.normal(size=3000) + (3 - 2j)
    cuts = [0, 700, 1500, 1501, 3000]
    offs, off = [], 0j
    for n in range(3000):
        if n in cuts:
            offs.append(off)
        off = off + (z[n] - off) * L
    gains, lens = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        g = 0j
        for n in range(a, b):
            g = g + (z[n] - g) * L
        gains.append(g)
        lens.append(b - a)
    for r in range(4):
        assert abs(sharding.iq_start_offset(gains, lens, lam, r) - offs[r]) < 1e-13


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    for p in (ROOT, os.path.join(ROOT, 'tests')):
        if p not in sys.path:
            sys.path.insert(0, p)
    import signals
    from oracle import oracle as orc
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        # ---------------- time segments (config 5 shape, 5 chunks over 2 ranks)
        kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True)
        body = signals.c1_bytes(5 * 32768, seed=5, header=False)
        start, cnt = sharding.segment_shard(5, world, rank)
        seg = body[start * CB:(start + cnt) * CB]
        ch = orc.Chain(**kw)
        ch.run(seg)                                           # pass 1: gain from a zero offset
        off0 = sharding.exchange_iq_gain(dist, torch, complex(ch._off[0]), cnt * 32768,
                                         1 - 50 / kw['fs'])
        ch2 = orc.Chain(**kw)
        ch2._off[0] = off0
        out = ch2.run(seg)                                    # pass 2 from the true start offset
        # ---------------- VFO rows (config 3 shape, 5 rows over 2 ranks), raw broadcast
        raw3, vf = signals.c3_bytes(2 * 32768, seed=3, k=4)
        t = torch.from_numpy(np.frombuffer(raw3, dtype=np.uint8).copy()) if rank == 0 else \
            torch.empty(len(raw3), dtype=torch.uint8)
        sharding.broadcast_raw(dist, torch, t, src=0)
        kw3 = dict(fs=2_400_000, enc='h', swap=True, center=0, dec=64, demod='fm', omega_out=5000,
                   simo=True, vfos=vf)
        full = orc.Chain(**kw3)
        lo, hi = sharding.row_shard(full.R, world, rank)
        mine = orc.Chain(**kw3)
        mine.rows = full.rows[lo:hi]
        mine.R = hi - lo
        mine.shift = orc.nco_table(mine.rows, mine.fs, mine.n, True)
        rows = mine.run(t.numpy().tobytes())
        q.put((rank, start, cnt, out, lo, hi, rows))
        dist.barrier()
    except BaseException as e:                                # surface the failure, do not hang the parent
        q.put((rank, repr(e)))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_gloo_matches_single_process():
    import signals
    from oracle import oracle as orc
    world, port = 2, _free_port()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    assert all(len(r) == 7 for r in res), res
    res.sort(key=lambda x: x[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    kw = dict(fs=1_024_000, enc='h', center=15000, dec=64, demod='fm', omega_out=5000, correct_iq=True)
    body = signals.c1_bytes(5 * 32768, seed=5, header=False)
    serial = orc.Chain(**kw).run(body)
    got = np.concatenate([r[3] for r in res], axis=1)
    assert got.shape == serial.shape
    assert np.max(np.abs(got - serial)) / np.max(np.abs(serial)) < 1e-12
    raw3, vf = signals.c3_bytes(2 * 32768, seed=3, k=4)
    kw3 = dict(fs=2_400_000, enc='h', swap=True, center=0, dec=64, demod='fm', omega_out=5000,
               simo=True, vfos=vf)
    serial3 = orc.Chain(**kw3).run(raw3)
    got3 = sharding.concat_rows([r[6] for r in res])
    assert got3.shape == serial3.shape and np.array_equal(got3, serial3)


def test_bank_grid_spends_ranks_on_rows_only_while_a_rank_keeps_enough_of_them():
    from sdrterm_b200.multigpu import bank_grid
    assert [bank_grid(17, w) for w in (1, 2, 4, 8)] == [(1, 1), (2, 1), (2, 2), (2, 4)]      # config 3
    assert [bank_grid(257, w) for w in (1, 2, 4, 8)] == [(1, 1), (2, 1), (4, 1), (8, 1)]     # config 4
    for rows in (1, 3, 17, 33, 257):
        for w in (1, 2, 4, 8):
            rg, tg = bank_grid(rows, w)
            assert rg * tg == w and (rg == 1 or rows // rg >= 8)


class _FakeEngine:
    """Stands in for the device engine: records what each call was given (host logic under test)."""
    log = []

    def __init__(self, plan, max_chunks=1, device=0, **kw):
        self.plan, self.max_chunks = plan, max_chunks
        self.iq_state = 0j

    def process(self, raw):
        raw = np.ascontiguousarray(raw).view(np.uint8).reshape(-1)
        _FakeEngine.log.append(raw.copy())
        n = raw.size // CB
        return np.zeros((1, n * self.plan.M))

    def iq_gain(self, raw):
        pass

    def close(self):
        pass


@pytest.mark.parametrize('nbytes', [7 * CB, 6 * CB + 1000, 3 * CB + 1])
def test_run_file_sharded_hands_every_rank_its_chunks_with_the_stale_tail(tmp_path, monkeypatch, nbytes):
    """Host logic of config 5 (no GPU): the segments of all ranks, in rank order, are exactly the
    chunks the reference's reused read buffer would present (SURVEY 8-Q5), offset by dataOffset."""
    from gpu_util import chunked
    from sdrterm_b200 import multigpu
    monkeypatch.setattr(multigpu, 'Engine', _FakeEngine)
    rng = np.random.default_rng(1)
    body = rng.integers(0, 256, nbytes, dtype=np.uint8).tobytes()
    path = tmp_path / 'in.raw'
    path.write_bytes(b'HEAD' * 10 + body)

    class FakeDist:
        def __init__(self, rank, world):
            self.rank, self.world = rank, world

        def get_world_size(self):
            return self.world

        def get_rank(self):
            return self.rank

    for world in (1, 2, 3):
        got = []
        for rank in range(world):
            _FakeEngine.log.clear()
            out = multigpu.run_file_sharded(str(path), None, fs=1_024_000, enc='h', dec=64, center=15000, omega_out=5000,
                                            data_offset=40, batch_chunks=2, device=0,
                                            dist=FakeDist(rank, world) if world > 1 else None, torch=torch)
            got += list(_FakeEngine.log)
            assert out.shape[1] % 512 == 0
        allb = np.concatenate(got) if got else np.zeros(0, dtype=np.uint8)
        assert np.array_equal(allb, chunked(body).reshape(-1)), (world, nbytes)


def _bank_worker(rank, world, port, q):
    """RowShardedBank (the product class) on two gloo ranks with a recording engine: the grid, the
    row slices and the double-buffered hand-over of the leader's raw batches."""
    for p in (ROOT, os.path.join(ROOT, 'tests')):
        if p not in sys.path:
            sys.path.insert(0, p)
    import ctypes
    from sdrterm_b200 import multigpu
    # the stand-in engine reads host memory: the product classes must keep their tensors on the
    # host, as they do on a machine without a CUDA device
    torch.cuda.is_available = lambda: False
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), SDRB_BCAST='nccl')
    dist.init_process_group('gloo', rank=rank, world_size=world)

    class Rec:
        seen = []

        def __init__(self, plan, max_chunks=1, device=0, **kw):
            self.plan, self.tc = plan, None

        def reserve_sms(self, n):
            pass

        def process_device(self, raw_ptr, nchunks, out_ptr, stream=0):
            nb = nchunks * self.plan.chunk_bytes
            Rec.seen.append(bytes((ctypes.c_uint8 * nb).from_address(raw_ptr)))

        def close(self):
            pass

    try:
        multigpu.Engine = Rec
        rows = [-200_000, -100_000, 100_000, 200_000, 0]
        bank = multigpu.RowShardedBank(2_400_000, 'h', 64, rows, 2, 0, dist, torch, min_rows=2, demod='fm', swap=True,
                                       omega_out=5000)
        rng = np.random.default_rng(11)
        data = [rng.integers(0, 256, 2 * CB, dtype=np.uint8) for _ in range(5)]
        batches = [torch.from_numpy(d.copy()) if rank == bank.leader else torch.empty(2 * CB, dtype=torch.uint8) for d in data]
        outs = [torch.empty((len(bank.rows), 2 * bank.M), dtype=torch.float64) for _ in data]
        bank.run(batches, 2, outs)
        bank.run(batches[:2], 1, outs[:2])                       # a shorter batch through the same buffers
        ok = [Rec.seen[i] == data[i].tobytes() for i in range(5)] + [Rec.seen[5 + i] == data[i][:CB].tobytes() for i in range(2)]
        q.put((rank, bank.row_groups, bank.time_groups, bank.lo, bank.hi, bank.transport, ok, len(Rec.seen)))
        dist.barrier()
    except BaseException as e:
        q.put((rank, repr(e)))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_row_sharded_bank_two_rank_gloo():
    world, port = 2, _free_port()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_bank_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    assert all(len(r) == 8 for r in res), res
    res.sort(key=lambda x: x[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert [(r[1], r[2]) for r in res] == [(2, 1), (2, 1)]
    assert [(r[3], r[4]) for r in res] == [(0, 3), (3, 5)]                 # balanced row slices, larger share first
    assert all(r[5] == 'nccl' for r in res)                                  # the collective transport (gloo here)
    assert all(all(r[6]) and r[7] == 7 for r in res), res                    # every rank saw the leader's bytes, in order


def test_bank_refuses_iq_correction_across_time_groups():
    """A bank on time groups has no IQ-offset hand-off: it must say so instead of restarting the
    corrector in every group."""
    from sdrterm_b200 import multigpu

    class FakeDist:
        def get_world_size(self):
            return 8

        def get_rank(self):
            return 3

    with pytest.raises(NotImplementedError):
        multigpu.RowShardedBank(2_400_000, 'h', 64, list(range(-8, 9)), 4, 0, FakeDist(), torch, correct_iq=True, demod='fm',
                                omega_out=5000)


def _chain_worker(rank, world, port, q):
    """TimeShardedChain (the product class) on gloo ranks with an engine stand-in that plays the
    device side of the IQ hand-off in numpy: export (gain, samples), all-gather, prefix."""
    for p in (ROOT, os.path.join(ROOT, 'tests')):
        if p not in sys.path:
            sys.path.insert(0, p)
    import ctypes
    from sdrterm_b200 import multigpu
    # the stand-in engine writes host memory: the product class must keep its tensors on the host,
    # as it does on a machine without a CUDA device
    torch.cuda.is_available = lambda: False
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    lam = 1 - 50 / 1_024_000

    class Plan:
        N, lam_ = 32768, lam

    class Eng:
        calls = []
        start = None

        def __init__(self, plan, max_chunks=1, device=0, **kw):
            pass

        def process_device(self, *a):
            Eng.calls.append('all')

        def process_device_phases(self, raw_ptr, nchunks, out_ptr, phases, stream=0):
            Eng.calls.append(phases)

        def iq_export_device(self, dst_ptr, nsamples, stream=0):
            g = complex(0.25 * (rank + 1), -0.5 * (rank + 1))          # what this segment "gained"
            d = (ctypes.c_double * 3).from_address(dst_ptr)
            d[0], d[1], d[2] = g.real, g.imag, float(nsamples)
            Eng.calls.append('export')

        def iq_prefix_device(self, gains_ptr, r, stream=0):
            d = np.array((ctypes.c_double * (3 * world)).from_address(gains_ptr))
            gains = [complex(d[3 * i], d[3 * i + 1]) for i in range(world)]
            lens = [int(d[3 * i + 2]) for i in range(world)]
            Eng.start = sharding.iq_start_offset(gains, lens, lam, r)
            Eng.calls.append('prefix')

        def close(self):
            pass

    try:
        multigpu.Engine = Eng
        chain = multigpu.TimeShardedChain(Plan(), 4, 0, dist, torch)
        chain.step(0, 3 + rank, 0)
        q.put((rank, Eng.calls, Eng.start))
        dist.barrier()
    except BaseException as e:
        q.put((rank, repr(e)))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_time_sharded_chain_three_rank_gloo():
    world, port = 3, _free_port()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_chain_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    assert all(len(r) == 3 for r in res), res
    res.sort(key=lambda x: x[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    lam = 1 - 50 / 1_024_000
    gains = [complex(0.25 * (r + 1), -0.5 * (r + 1)) for r in range(world)]
    lens = [(3 + r) * 32768 for r in range(world)]
    off = 0j
    for r in range(world):
        # front end + gain from zero (MAIN | IQSCAN | ZERO_IQ), export, all-gather, prefix, IQSCAN | FINISH
        assert res[r][1] == [1 | 2 | 8, 'export', 'prefix', 2 | 4]
        assert abs(res[r][2] - off) < 1e-15                      # the offset entering segment r
        off = lam ** lens[r] * off + gains[r]
