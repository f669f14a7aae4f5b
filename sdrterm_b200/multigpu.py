"""Multi-GPU drivers of the chain: one process per GPU, ``torch.distributed`` for the plumbing
(NCCL on the GPU box, gloo in the CPU tests of the host logic).  The path shards two ways
(SURVEY 8e) and needs at most one small exchange:

* ``TimeShardedChain`` -- offline files (BASELINE config 5).  Chunks are independent except for
  the IQ corrector's complex offset (reference src/misc/read_file.py:53), an affine recurrence
  ``off' = lam off + L z``.  Every rank owns one contiguous time segment on chunk boundaries,
  runs its block front end from a zero offset, the ranks all-gather the offset each segment
  *gained* (3 doubles per rank, on the stream, no host round trip), every rank folds the gains of
  the segments before it into its start offset and finishes.  The raw data is read once.
* ``RowShardedBank`` -- ``--simo`` banks (configs 3/4; reference src/dsp/vfo_processor.py:42-48,
  80-84: rows are independent given the raw chunk and go to separate sockets).  Ranks form a
  (row group x time group) grid (``bank_grid``): rows are dealt out contiguously and evenly inside
  a row group, and the leader's raw batch reaches the other ranks of its group as raw BYTES
  (2*itemsize bytes per sample, not 16) through an NCCL broadcast that is pipelined against the
  kernels of the previous batch; nothing is gathered, each rank frames its own rows.  A wide bank
  (config 4: 257 rows) is all row groups; a narrow one (config 3: 17 rows) uses two row groups and
  spends the remaining ranks on time segments, because every rank of a row group must receive
  every byte of the segment and NVLink ingress, not the kernels, would otherwise be the limit.

``run_file_sharded`` is the product entry point for config 5; bench.py drives the same classes.
"""
from __future__ import annotations

import os

import numpy as np

from . import sharding
from .engine import Engine
from .plan import Plan, build_plan

CHUNK_BYTES = 131072


def bind_to_gpu_numa_node(device: int) -> bool:
    """Pin the calling process to the CPUs closest to ``device`` (NVML's ideal affinity) BEFORE it
    allocates page-locked staging memory: pinned pages then live on the GPU's own NUMA node and the
    H2D / D2H DMA does not cross the socket interconnect.  torchrun does not do this, and with eight
    ranks streaming from host memory it decides the end-to-end rate.  Returns False when NVML is
    unavailable (nothing is changed then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(device))
        return True
    except Exception:
        return False


SEAMLESS_REFUSAL = ('seamless mode is single-GPU: time segments would need a halo of D chunks (the '
                    'lookahead) and a hand-off of the forward filter state between ranks, which is not '
                    'built yet')


class TimeShardedChain:
    """One rank's share of a time-segment sharded stream.  ``step`` processes one device-resident
    segment of ``nchunks`` chunks; with world == 1 it is a plain ``process_device``."""

    def __init__(self, plan: Plan, max_chunks: int, device: int, dist=None, torch=None):
        if getattr(plan, 'seamless', False):
            raise ValueError(SEAMLESS_REFUSAL)
        self.plan, self.dist, self.torch = plan, dist, torch
        self.world = dist.get_world_size() if dist is not None else 1
        self.rank = dist.get_rank() if dist is not None else 0
        self.engine = Engine(plan, max_chunks=max_chunks, device=device)
        if self.world > 1:
            # (CPU tensors only when there is no CUDA device at all: the gloo tests of this host logic)
            dev = torch.device('cuda', device) if torch.cuda.is_available() else torch.device('cpu')
            self._mine = torch.zeros(3, dtype=torch.float64, device=dev)
            self._all = torch.zeros(3 * self.world, dtype=torch.float64, device=dev)

    def step(self, raw_ptr: int, nchunks: int, out_ptr: int, stream: int = 0) -> None:
        e = self.engine
        if self.world == 1:
            e.process_device(raw_ptr, nchunks, out_ptr, stream)
            return
        nsamp = nchunks * self.plan.N
        # block front end + the offset this segment gains from zero; exchange; finish
        e.process_device_phases(raw_ptr, nchunks, 0, 1 | 2 | 8, stream)
        e.iq_export_device(self._mine.data_ptr(), nsamp, stream)
        self.dist.all_gather_into_tensor(self._all, self._mine)
        e.iq_prefix_device(self._all.data_ptr(), self.rank, stream)
        e.process_device_phases(raw_ptr, nchunks, out_ptr, 2 | 4, stream)

    def close(self):
        self.engine.close()


def bank_grid(nrows: int, world: int, min_rows: int = 8) -> tuple[int, int]:
    """(row_groups, time_groups) with row_groups * time_groups == world.  Every rank of a row group
    needs every raw byte of its time segment, so a rank's NVLink ingress is 2*itemsize bytes per
    input sample whatever the number of row groups: splitting a narrow bank over many ranks makes
    the broadcast, not the kernels, the limit (17 rows over 8 ranks: 2 rows of compute per 4 bytes
    received).  Ranks are therefore spent on rows only while a rank keeps >= ``min_rows`` rows, and
    on time segments beyond that -- a segment's bytes then reach world/time_groups ranks only."""
    rg = 1
    while rg * 2 <= world and world % (rg * 2) == 0 and nrows // (rg * 2) >= min_rows:
        rg *= 2
    return rg, world // rg


class PeerFanout:
    """The raw batch of a time group's leader -> every other rank of the group through NVLink peer
    memory, driven by the leader's copy engines (no SM is taken from the kernels that run beside
    it; an ``ncclBroadcast`` of the same bytes costs the 17-row bank 25 % of its rate at two GPUs).

    Every rank of the group allocates ``NBUF`` = 3 slots of symmetric memory
    (``torch.distributed._symmetric_memory``: cuMem allocations mapped into every rank's address
    space, so a peer slot is an ordinary local-device tensor and ``copy_`` is one D2D memcpy over
    NVLink; measured 695 GB/s to one peer against 29 GB/s through legacy CUDA-IPC handles,
    microbench/peer_copy.py).  Batch i: the leader copies its bytes into slot i % 3 of every peer
    (one stream per peer), then all ranks of the group meet in a one-word all-reduce D_i on their
    side streams.  A receiver lets D_i start only when its kernels of batch i-2 are done, so on the
    leader "D_i complete" means slot (i+1) % 3 is free everywhere, and on a receiver it means batch
    i has landed.  With three slots D_i does not have to wait for the kernels of batch i-1, so its
    latency stays off the critical path; the copy of batch i+1 overlaps the kernels of batch i."""

    NBUF = 3

    def __init__(self, dist, torch, group, ranks, leader: int, nbytes: int, device: int):
        import torch.distributed._symmetric_memory as symm
        self.dist, self.torch, self.group = dist, torch, group
        self.is_leader = dist.get_rank() == leader
        dev = torch.device('cuda', device)
        self.nbytes = nbytes
        self.mem = symm.empty(self.NBUF * nbytes, dtype=torch.uint8, device=dev)
        hdl = symm.rendezvous(self.mem, group)
        self.bufs = [self.mem[k * nbytes:(k + 1) * nbytes] for k in range(self.NBUF)]
        self.peers = []                                   # leader: [peer][slot] views of the peers' slots
        if self.is_leader:
            for gr in range(len(ranks)):
                if ranks[gr] != leader:
                    view = hdl.get_buffer(gr, (self.NBUF, nbytes), torch.uint8)
                    self.peers.append([view[k] for k in range(self.NBUF)])
        self._hdl = hdl
        self.side = torch.cuda.Stream(device=dev)
        self.lanes = [torch.cuda.Stream(device=dev) for _ in self.peers]
        self.flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self.read_done = [None] * self.NBUF               # receiver: event after the kernels that read the slot
        self.last = None

    def begin(self) -> None:
        """Start of a sequence of batches (numbered from 0 again): every rank's earlier kernels
        are done before the leader may overwrite a slot."""
        torch = self.torch
        self.side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.side):
            self.last = self.dist.all_reduce(self.flag, group=self.group, async_op=True)
        self.read_done = [None] * self.NBUF

    def post(self, i: int, src, nbytes: int):
        """Start batch i on its way; returns the work object of D_i (wait() on the compute stream)."""
        torch = self.torch
        cur = torch.cuda.current_stream()
        slot = i % self.NBUF
        if self.is_leader:
            for lane, peer in zip(self.lanes, self.peers):
                lane.wait_stream(cur)                     # the source batch is ready
                with torch.cuda.stream(lane):
                    if self.last is not None:
                        self.last.wait()                  # D_{i-1}: the slot is free on every peer
                    peer[slot][:nbytes].copy_(src[:nbytes], non_blocking=True)
                self.side.wait_stream(lane)
        else:
            ev = self.read_done[(i - 2) % self.NBUF] if i >= 2 else None
            if ev is not None:
                self.side.wait_event(ev)
        with torch.cuda.stream(self.side):
            self.last = self.dist.all_reduce(self.flag, group=self.group, async_op=True)
        return self.last

    def slot(self, i: int):
        return self.bufs[i % self.NBUF]

    def consumed(self, i: int) -> None:
        """The kernels that read batch i have been enqueued on the current stream."""
        if not self.is_leader:
            ev = self.torch.cuda.Event()
            ev.record(self.torch.cuda.current_stream())
            self.read_done[i % self.NBUF] = ev


class RowShardedBank:
    """One rank's share of a ``--simo`` bank on a (row group x time group) grid of ranks.
    ``rows_hz`` is the full bank (the listed VFO offsets + the centre, reference
    vfo_processor.py:42-46); rank (tg, rg) owns the rg-th balanced slice of the rows for the
    tg-th time segment and builds a plan for its slice only.  ``run(batches)`` processes a
    sequence of raw batches that exist on the time group's leader (rg == 0); batch i+1 travels to
    the group (``PeerFanout``; ``SDRB_BCAST=nccl`` selects a plain NCCL broadcast instead) while
    the kernels of batch i run.  Nothing is gathered: each rank frames its own rows (one socket
    per row, vfo_processor.py:80-84)."""

    def __init__(self, fs: int, enc: str, dec: int, rows_hz, max_chunks: int, device: int, dist=None, torch=None,
                 min_rows: int | None = None, **plan_kw):
        if plan_kw.get('seamless'):
            raise ValueError(SEAMLESS_REFUSAL)
        self.dist, self.torch = dist, torch
        self.world = dist.get_world_size() if dist is not None else 1
        self.rank = dist.get_rank() if dist is not None else 0
        self.rows_all = [int(f) for f in rows_hz]
        if min_rows is None:
            min_rows = 8
        self.row_groups, self.time_groups = bank_grid(len(self.rows_all), self.world, min_rows)
        if plan_kw.get('correct_iq') and self.time_groups > 1:
            # the corrector's offset runs through the whole stream (read_file.py:53): time groups
            # would each start from their own state.  TimeShardedChain has the hand-off; a bank does
            # not (BASELINE configs 3 and 4 run without --correct-iq), so it must not pretend to.
            raise NotImplementedError('--correct-iq on a bank spread over time groups needs the IQ-offset hand-off: '
                                      f'use min_rows <= {max(1, len(self.rows_all) // self.world)} (row groups only)')
        self.tg, self.rg = divmod(self.rank, self.row_groups)
        self.lo, self.hi = sharding.row_shard(len(self.rows_all), self.row_groups, self.rg)
        self.rows = self.rows_all[self.lo:self.hi]
        self.leader = self.tg * self.row_groups               # global rank that holds the segment's raw bytes
        self.max_chunks = max_chunks
        self.plan = build_plan(fs, enc, dec, self.rows, simo=True, **plan_kw)
        self.engine = Engine(self.plan, max_chunks=max_chunks, device=device)
        self.chunk_bytes = self.plan.chunk_bytes
        self.group = None
        self.fanout = None
        self.transport = 'none'
        if self.row_groups > 1:
            # every rank creates every group (torch.distributed requires it), keeps its own
            for t in range(self.time_groups):
                g = dist.new_group(list(range(t * self.row_groups, (t + 1) * self.row_groups)))
                if t == self.tg:
                    self.group = g
            # (CPU tensors only when there is no CUDA device at all: the gloo tests of this host logic)
            dev = torch.device('cuda', device) if torch.cuda.is_available() else torch.device('cpu')
            ranks = list(range(self.leader, self.leader + self.row_groups))
            nbytes = max_chunks * self.chunk_bytes
            want = os.environ.get('SDRB_BCAST', 'peer')
            ok = torch.zeros(1, dtype=torch.int32, device=dev)
            if want == 'peer':
                try:
                    self.fanout = PeerFanout(dist, torch, self.group, ranks, self.leader, nbytes, device)
                    ok += 1
                except Exception as ex:                       # no symmetric memory / peer access on this box
                    import sys
                    print(f'sdrterm_b200: peer-memory fan-out unavailable ({ex!r}); using ncclBroadcast', file=sys.stderr)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)         # one transport for everybody
            if int(ok.item()) == 1:
                self.transport = 'peer'
                # the one-word all-reduce that paces the copies needs a free SM while the persistent
                # kernels of the previous batch are still running, or it sits between two batches
                self.engine.reserve_sms(int(os.environ.get('SDRB_PEER_SMS', '2')))
            else:
                self.fanout = None
                self.transport = 'nccl'
                # the broadcast runs beside this batch's kernels on SMs: leave it some
                self.engine.reserve_sms(int(os.environ.get('SDRB_BCAST_SMS', '8')))
                self._bufs = [torch.empty(nbytes, dtype=torch.uint8, device=dev) for _ in range(2)]

    @property
    def M(self) -> int:
        return self.plan.M

    @property
    def W(self) -> int:
        """Doubles per chunk and row of the output (2M for iq)."""
        return self.plan.W

    def _post(self, i: int, src, nbytes: int):
        """Start batch i on its way to the ranks of the time group."""
        if self.row_groups == 1:
            return None
        if self.fanout is not None:
            return self.fanout.post(i, src, nbytes)
        b = self._bufs[i & 1][:nbytes]
        if self.rank == self.leader:
            b.copy_(src[:nbytes], non_blocking=True)
        return self.dist.broadcast(b, src=self.leader, group=self.group, async_op=True)

    def run(self, batches, nchunks: int, outs, stream: int = 0) -> None:
        """``batches``: list of uint8 device tensors (on the leader; elsewhere only the count
        matters); ``outs``: list of (rows, nchunks*W) float64 device tensors of this rank.  The
        kernels go to ``stream``, which must be the current torch stream."""
        n = len(batches)
        if nchunks > self.max_chunks or len(outs) < n:
            raise ValueError(f'{nchunks} chunks per batch exceed max_chunks = {self.max_chunks}, or too few output tensors')
        nbytes = nchunks * self.chunk_bytes
        if self.fanout is not None:
            self.fanout.begin()
        w = self._post(0, batches[0], nbytes)
        for i in range(n):
            if w is not None:
                w.wait()
            w = self._post(i + 1, batches[i + 1], nbytes) if i + 1 < n else None
            if self.row_groups == 1 or (self.fanout is not None and self.rank == self.leader):
                src = batches[i]
            elif self.fanout is not None:
                src = self.fanout.slot(i)
            else:
                src = self._bufs[i & 1]
            self.engine.process_device(src.data_ptr(), nchunks, outs[i].data_ptr(), stream)
            if self.fanout is not None:
                self.fanout.consumed(i)

    def close(self):
        self.engine.close()


def run_file_sharded(path: str, out_path: str | None, *, fs: int, enc: str, dec: int, center: int = 0,
                     demod: str = 'fm', omega_out: int = 12500, correct_iq: bool = False, swap: bool = False,
                     data_offset: int = 0, batch_chunks: int = 2048, device: int | None = None, dist=None,
                     torch=None, seamless: bool = False) -> np.ndarray | None:
    """BASELINE config 5: an offline IQ file, time-segment sharded over the ranks of ``dist``
    (``None`` = single process).  Every rank reads ITS segment of the file (whole 131072-byte
    chunks counted from ``data_offset``; the reference's stale-tail chunk, SURVEY 8-Q5, belongs to
    the last rank), runs an IQ-gain pre-pass over it when ``correct_iq`` (raw bytes only, no
    outputs), exchanges the gains, then demodulates its segment batch by batch through the
    double-buffered host path.  Rank r writes ``out_path + '.part%04d' % r`` (or returns the array
    when ``out_path`` is None): the concatenation in rank order is the reference's output file.
    ``seamless=True`` is refused (ValueError): see SEAMLESS_REFUSAL."""
    if seamless:
        raise ValueError(SEAMLESS_REFUSAL)
    if torch is None:
        import torch as _t
        torch = _t
    world = dist.get_world_size() if dist is not None else 1
    rank = dist.get_rank() if dist is not None else 0
    if device is None:
        device = int(os.environ.get('LOCAL_RANK', '0'))
    size = os.path.getsize(path) - data_offset
    nchunks_total = -(-size // CHUNK_BYTES)
    first, count = sharding.segment_shard(nchunks_total, world, rank)
    plan = build_plan(fs, enc, dec, [center], swap=swap, correct_iq=correct_iq, demod=demod, omega_out=omega_out)
    eng = Engine(plan, max_chunks=batch_chunks, device=device)

    def read_segment():
        """This rank's chunks as the reference's reused read buffer presents them."""
        with open(path, 'rb') as fh:
            fh.seek(data_offset + first * CHUNK_BYTES)
            raw = np.frombuffer(fh.read(count * CHUNK_BYTES), dtype=np.uint8)
            if raw.size < count * CHUNK_BYTES:           # short final read: stale tail of the chunk before
                full = np.empty(count * CHUNK_BYTES, dtype=np.uint8)
                full[:raw.size] = raw
                tail0 = raw.size - (raw.size % CHUNK_BYTES)
                short = raw.size - tail0
                if tail0 >= CHUNK_BYTES:
                    prev = raw[tail0 - CHUNK_BYTES:tail0]
                elif first > 0:
                    fh.seek(data_offset + (first + count - 2) * CHUNK_BYTES)
                    prev = np.frombuffer(fh.read(CHUNK_BYTES), dtype=np.uint8)
                else:
                    prev = np.zeros(CHUNK_BYTES, dtype=np.uint8)
                full[tail0 + short:] = prev[short:]
                raw = full
        return raw

    raw = read_segment() if count else np.zeros(0, dtype=np.uint8)
    if correct_iq and world > 1:
        # pass 1: the offset this segment gains from a zero start (bytes only)
        eng.iq_state = 0j
        for b0 in range(0, count, batch_chunks):
            n = min(batch_chunks, count - b0)
            eng.iq_gain(raw[b0 * CHUNK_BYTES:(b0 + n) * CHUNK_BYTES])
        gain = eng.iq_state
        start = sharding.exchange_iq_gain(dist, torch, gain, count * plan.N, plan.lam,
                                          device=torch.device('cuda', device) if dist.get_backend() == 'nccl' else None)
        eng.iq_state = start
    out = np.empty((1, count * plan.W), dtype=np.float64)
    for b0 in range(0, count, batch_chunks):
        n = min(batch_chunks, count - b0)
        out[:, b0 * plan.W:(b0 + n) * plan.W] = eng.process(raw[b0 * CHUNK_BYTES:(b0 + n) * CHUNK_BYTES])
    eng.close()
    if out_path is None:
        return out
    with open(out_path + '.part%04d' % rank, 'wb') as fh:
        fh.write(out[0].tobytes())
    return None
