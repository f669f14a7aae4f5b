#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 demodulation chain (see the contract in DESIGN.md).

Metric (BASELINE.json): input Msamples/s through the single-VFO FM chain, -d 64.
Workload at every N: configuration 1/5 of BASELINE.json -- int16 IQ at 1.024 MS/s,
`-c 15k -w 5k -d 64 --correct-iq -m fm` -- 2^28 complex samples (8192 chunks of 131072 bytes,
1 GiB of raw input) per GPU per step; for N > 1 the stream is time-segment sharded (one
contiguous segment per rank, IQ-corrector state handed off through an all-gather, weak scaling).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference ...                     # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's output

`--dump-outputs DIR` writes DIR/out.npy (float64): what the timed path returned in its last timed
step, the whole stream in rank order, or a fixed seeded sample of its columns beyond 64 MB.  The
inputs depend only on the arguments, so two builds can be compared output for output.

`--steps` is the number of timed steps of the headline measurement (`value`, `ms_per_step`,
`gpu_launches`; the reference arm likewise).  The secondary legs keep their own counts: `e2e`
times min(--steps, 3) steps, `simo` 24 batches and `simo_config4` 12.

One JSON line on stdout (rank 0).  `value`: device-resident input, CUDA-event timed, max over
ranks.  `e2e`: the same through the C ABI's host entry points (pinned host buffers, H2D and D2H
inside the timed region, double-buffered).  `roofline`: k_main's algorithmic bytes over its
CUDA-event duration vs the measured HBM copy bandwidth.  `cpu_baseline`: the oracle port on this
box's host cores over a bounded sample.  `simo`: config 3 (16 VFOs + centre, 17 rows) measured the
same way, rows sharded across ranks with an NCCL broadcast of each raw batch.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'tests')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

CB = 131072
FS, CENTER, OMEGA, DEC = 1_024_000, 15_000, 5_000, 64
METRIC = 'input Msamples/s through FM chain (d=64)'
WORKLOAD = ('config 1/5: single-VFO FM chain, int16 IQ, fs 1.024 MS/s, -c 15k -w 5k -d 64 '
            '--correct-iq, 2^28 samples (8192 chunks) per GPU per step')


# ------------------------------------------------------------------------------ CPU (oracle) arm
def cpu_chain_rate(nchunks_hint: int, target_s: float, nthreads: int):
    """Time the oracle port (decode + IQ + NCO + decimate + fm + LPF + pack) on host cores over
    a bounded sample of the same synthetic workload.  Returns (Msamples/s, sample description)."""
    import numpy as np
    import signals
    from oracle import oracle as orc
    kw = dict(fs=FS, enc='h', center=CENTER, dec=DEC, demod='fm', omega_out=OMEGA, correct_iq=True,
              nthreads=nthreads)
    base = signals.c1_bytes(16 * 32768, seed=0, header=False)

    def run(nch):
        body = (base * (-(-nch // 16)))[:nch * CB]
        ch = orc.Chain(**kw)
        t0 = time.perf_counter()
        out = ch.run_fast(body)
        _ = np.ascontiguousarray(out[0], dtype='=f8').tobytes()
        return time.perf_counter() - t0

    run(8)                                     # warm-up (library load, page faults)
    t = run(nchunks_hint)
    nch = int(max(nchunks_hint, min(16384, nchunks_hint * target_s / max(t, 1e-3))))
    best = min(run(nch) for _ in range(2))
    return nch * 32768 / best / 1e6, f'{nch} chunks ({nch * 32768} samples) of the workload, best of 2'


def host_threads() -> int:
    """Cores this process may use.  torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm
    passes its thread count to the oracle explicitly, so that setting never caps it."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def python_reference_rate(nch: int):
    """The UNMODIFIED Python reference (vendored by oracle/make_ref.py into oracle/_ref, git-ignored,
    shipped with the snapshot) timed in-process the way BASELINE.md section 3 describes: decode +
    IQ correction (read_file.py:100-103) -> DspProcessor._processChunk -> struct.pack, one thread
    (scipy's _sosfilt and the numba gufuncs are single-threaded).  None when _ref is absent."""
    ref = os.path.join(ROOT, 'oracle', '_ref', 'src')
    if not os.path.isdir(os.path.join(ref, 'dsp')):
        return None
    import numpy as np
    import signals
    os.environ.setdefault('NUMBA_CACHE_DIR', '/tmp/sdrb_numba_cache')
    sys.path.insert(0, ref)
    try:
        from struct import pack
        from dsp.dsp_processor import DspProcessor
        p = DspProcessor(FS, center=CENTER, omegaOut=OMEGA, dec=DEC, fileInfo={'bitsPerSample': np.dtype('<i2')})
        p.selectOutputFm()
        body = signals.c1_bytes(nch * 32768, seed=0, header=False)
        L = 50 / FS
        off = 0j
        N = 32768
        p._generateShift(N)
        x = np.empty((1, N), dtype=np.complex128)
        y = np.empty((1, N // DEC), dtype=np.complex128)
        z = np.empty((1, N // DEC), dtype=np.float64)

        import numba

        @numba.njit(cache=False, fastmath=True)
        def correct_iq(data, st, ind):                   # read_file.py:67-77, compiled as the reference compiles it
            for i in range(data.shape[0]):
                data[i] -= st[0]
                st[0] += data[i] * ind

        off = np.zeros(1, dtype=np.complex128)

        def chunk(c):
            v = np.frombuffer(body, dtype=[('re', '<i2'), ('im', '<i2')], count=N, offset=c * CB)
            zz = v['re'] + 1j * v['im']                  # read_file.py:101
            correct_iq(zz, off, L)
            x[0, :] = zz
            p._processChunk(x, y, z)                     # dsp_processor.py:140-149
            return pack('@' + (z.size * 'd'), *z.flat)   # dsp_processor.py:162

        chunk(0)                                        # numba JIT warm-up
        off[0] = 0
        t0 = time.perf_counter()
        for c in range(nch):
            chunk(c)
        dt = time.perf_counter() - t0
        return {'value': nch * N / dt / 1e6, 'unit': 'Msamples/s', 'cores': 1, 'kind': 'reference',
                'sample': f'{nch} chunks ({nch * N} samples), unmodified src/dsp from oracle/_ref, in-process'}
    except Exception as e:                               # missing numba etc.: report, do not fail the arm
        return {'unavailable': f'{type(e).__name__}: {e}'}
    finally:
        sys.path.remove(ref)


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import oracle as orc
    nthreads = host_threads()
    import numpy as np
    import signals
    kw = dict(fs=FS, enc='h', center=CENTER, dec=DEC, demod='fm', omega_out=OMEGA, correct_iq=True,
              nthreads=nthreads)
    nch = args.ref_chunks
    base = signals.c1_bytes(16 * 32768, seed=0, header=False)
    body = (base * (-(-nch // 16)))[:nch * CB]
    times = []
    for it in range(args.warmup + args.steps):
        ch = orc.Chain(**kw)
        t0 = time.perf_counter()
        out = ch.run_fast(body)
        _ = np.ascontiguousarray(out[0], dtype='=f8').tobytes()
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {'out': out})
    t = sum(times) / len(times)
    val = nch * 32768 / t / 1e6
    sample = f'{nch} chunks ({nch * 32768} samples) per step'
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'Msamples/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': t * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'note': 'value = the oracle port (oracle/, numpy + C restatement of src/dsp + SciPy '
                       'recurrences) on every host core: the conservative comparison; reference_python = the '
                       'unmodified Python reference vendored into oracle/_ref, one thread by construction'},
            'cpu_baseline': {'value': val, 'unit': 'Msamples/s', 'cores': nthreads, 'kind': 'port',
                             'sample': sample},
            'reference_python': python_reference_rate(64),
            'e2e': {'value': val, 'unit': 'Msamples/s', 'h2d_bytes_per_step': 0,
                    'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    emit(line)


# ------------------------------------------------------------------------------ clocks sampler
class Clocks:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                 '--format=csv,noheader,nounits', '-lms', '20'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                                    'sw_power_cap'), r[4:8]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx or None,
                'reasons': sorted(reasons), 'samples': len(sm),
                'window': 'nvidia-smi -lms 20 over warm-up, the timed steps and the identical profiled steps that follow'}


# ------------------------------------------------------------------------------ synthetic input
def synth_c1_device(torch, nsamples: int, seed: int, device):
    """Config-1 signal generated on the device (not timed): FM carrier at +15 kHz, 1 kHz tone,
    +-2.5 kHz deviation, amplitude 8000, AWGN sigma 200, DC (+37,-21), rounded to int16 I,Q."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((nsamples, 2), dtype=torch.int16, device=device)
    step = 1 << 22
    for s in range(0, nsamples, step):
        n = min(step, nsamples - s)
        t = (torch.arange(s, s + n, device=device, dtype=torch.float64)) / FS
        ph = 2 * torch.pi * 15_000 * t + 2.5 * torch.sin(2 * torch.pi * 1_000 * t)
        re = 8000.0 * torch.cos(ph) + 200.0 * torch.randn(n, generator=g, device=device, dtype=torch.float64) + 37.0
        im = 8000.0 * torch.sin(ph) + 200.0 * torch.randn(n, generator=g, device=device, dtype=torch.float64) - 21.0
        out[s:s + n, 0] = torch.clamp(torch.round(re), -32768, 32767).to(torch.int16)
        out[s:s + n, 1] = torch.clamp(torch.round(im), -32768, 32767).to(torch.int16)
    return out.view(torch.uint8).reshape(-1)


def synth_c3_device(torch, nsamples: int, seed: int, device, offs):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    fs = 2_400_000
    out = torch.empty((nsamples, 2), dtype=torch.int16, device=device)
    step = 1 << 21
    for s in range(0, nsamples, step):
        n = min(step, nsamples - s)
        t = (torch.arange(s, s + n, device=device, dtype=torch.float64)) / fs
        re = 100.0 * torch.randn(n, generator=g, device=device, dtype=torch.float64)
        im = 100.0 * torch.randn(n, generator=g, device=device, dtype=torch.float64)
        for i, f in enumerate(list(offs) + [0]):
            ph = 2 * torch.pi * f * t + (2000.0 / (700 + 40 * i)) * torch.sin(2 * torch.pi * (700 + 40 * i) * t) + 0.37 * i
            re += 1500.0 * torch.cos(ph)
            im += 1500.0 * torch.sin(ph)
        out[s:s + n, 0] = torch.clamp(torch.round(re), -32768, 32767).to(torch.int16)
        out[s:s + n, 1] = torch.clamp(torch.round(im), -32768, 32767).to(torch.int16)
    # big-endian on the wire (config 3): swap the two bytes of every int16
    b = out.view(torch.uint8).reshape(-1, 2)
    return b.flip(1).contiguous().reshape(-1)


# ------------------------------------------------------------------------------ CLI end to end
def measure_cli(torch, raw_dev, nch_small: int, nch_big: int):
    """file -> the drop-in CLI -> file, config 1 flags.  `wall` is what a user sees for the big file
    from a fresh `python -m sdrterm` process (interpreter start, CUDA context, plan tables from the
    on-disk cache, the run), best of two; `startup` is the same for a 64-chunk file.  The CUDA
    context alone takes 0.9-1.6 s and varies by more than the 0.3 s a GiB streams in, so the
    streaming rate is not the difference of two process times: `steady` times the CLI's own
    `main(argv)` in THIS process (context already up) on the big file, best of two -- the same
    reader thread, page-locked chunk pool, processor and file writer, minus process start."""
    import shutil
    import tempfile
    import signals
    res = {}
    d = '/dev/shm' if os.path.isdir('/dev/shm') else tempfile.gettempdir()
    # the CLI caches its plan tables; keep that cache out of the (possibly read-only) source tree
    plan_cache = tempfile.mkdtemp(prefix='sdrb_plan_cache_')
    saved_cache = os.environ.get('SDRB_PLAN_CACHE')
    os.environ['SDRB_PLAN_CACHE'] = plan_cache
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, 'src'))
    times = {}
    flags = ['-c', '15k', '-w', '5k', '-d', '64', '--correct-iq']
    made = []

    def make(nch):
        fin = os.path.join(d, f'sdrb_cli_in_{os.getpid()}_{nch}.wav')
        fout = os.path.join(d, f'sdrb_cli_out_{os.getpid()}_{nch}.bin')
        body = raw_dev[:nch * CB].cpu().numpy().tobytes()
        with open(fin, 'wb') as fh:
            fh.write(signals.wav_header(FS, 16, len(body)) + body)
        made.extend([fin, fout])
        return fin, fout

    try:
        for nch in (64, nch_big, 64, nch_big):       # the first, tiny run pays the cold start (plan cache); then best of 2
            fin, fout = make(nch)
            t0 = time.perf_counter()
            # the CLI is its own process: it starts with the machine's full CPU set, not this rank's
            # NUMA binding
            unbind = (lambda: os.sched_setaffinity(0, _ALL_CPUS)) if _ALL_CPUS else None
            r = subprocess.run([sys.executable, '-m', 'sdrterm', '-i', fin, '-o', fout] + flags, env=env, cwd=d,
                               capture_output=True, text=True, timeout=600, preexec_fn=unbind)
            times[nch] = min(times.get(nch, 1e9), time.perf_counter() - t0)
            nout = os.path.getsize(fout) if os.path.exists(fout) else 0
            if r.returncode != 0 or nout < nch * 512 * 8:
                return {'unavailable': f'cli exit {r.returncode}, {nout} bytes out: {r.stderr[-300:]}'}
        from sdrterm_b200 import sdrterm as cli
        fin, fout = make(nch_big)
        t_in = 1e9
        import contextlib
        import io
        for _ in range(3):
            t0 = time.perf_counter()
            with contextlib.redirect_stderr(io.StringIO()):
                cli.main(['-i', fin, '-o', fout] + flags)
            t_in = min(t_in, time.perf_counter() - t0)
        if os.path.getsize(fout) < nch_big * 512 * 8:
            return {'unavailable': 'in-process main() wrote a short file'}
        res = {'wall_msps': nch_big * 32768 / times[nch_big] / 1e6,
               'steady_msps': nch_big * 32768 / t_in / 1e6,
               'seconds': {'process_64_chunks': times[64], f'process_{nch_big}_chunks': times[nch_big],
                           f'main_in_process_{nch_big}_chunks': t_in},
               'chunks': nch_big,
               'note': 'python -m sdrterm -i <wav> -o <file> -c 15k -w 5k -d 64 --correct-iq, files on tmpfs; '
                       'wall = fresh process, steady = the same main(argv) called in this process'}
    except Exception as e:
        res = {'unavailable': f'{type(e).__name__}: {e}'}
    finally:
        for f in made:
            if os.path.exists(f):
                os.unlink(f)
        if saved_cache is None:
            os.environ.pop('SDRB_PLAN_CACHE', None)
        else:
            os.environ['SDRB_PLAN_CACHE'] = saved_cache
        shutil.rmtree(plan_cache, ignore_errors=True)
    return res


# ------------------------------------------------------------------------------ CUDA arm
def measure_e2e(torch, Engine, pl, raw, sub, e2e_ch, local, args, barrier, max_over_ranks, world):
    """Host pinned buffers through sdrb_submit / sdrb_wait, H2D and D2H inside the timed region."""
    eng2 = Engine(pl, max_chunks=sub, device=local)
    host_raw = torch.empty(e2e_ch * CB, dtype=torch.uint8).pin_memory()
    host_raw.copy_(raw[:e2e_ch * CB].cpu())
    nb = -(-e2e_ch // sub)
    host_out = [torch.empty(sub * pl.M, dtype=torch.float64).pin_memory() for _ in range(2)]

    def step_e2e():
        pend = [None, None]
        for b in range(nb):
            s = b & 1
            if pend[s] is not None:
                eng2.wait(s)
            n = min(sub, e2e_ch - b * sub)
            eng2.submit(s, host_raw.data_ptr() + b * sub * CB, n, host_out[s].data_ptr())
            pend[s] = n
        eng2.wait(0)
        eng2.wait(1)

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    return world * e2e_ch * 32768 * e2e_steps / dt / 1e6



def run_cuda_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sdrterm_b200.engine import Engine
    from sdrterm_b200.plan import build_plan
    from sdrterm_b200 import multigpu

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the CUDA arm has no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    global _ALL_CPUS
    _ALL_CPUS = os.sched_getaffinity(0) if hasattr(os, 'sched_getaffinity') else None
    numa_bound = multigpu.bind_to_gpu_numa_node(local) if not args.no_numa else False
    numa_cpus = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else None
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=180))
    if world != args.gpus and rank == 0:
        print(f'# note: --gpus {args.gpus} but WORLD_SIZE {world}', file=sys.stderr)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    _align = [None]

    def align_on_device():
        """N > 1: a one-word all-reduce on the stream right before the start event.  The ranks'
        host threads leave the barrier up to a millisecond apart; without this the early ranks'
        start events precede the late rank's first kernel, and the skew is charged to a timed
        window that is only a few milliseconds long.  With it every rank's start event sits at the
        same point of the device timeline; the timed region itself is unchanged (K steps)."""
        if world > 1:
            if _align[0] is None:
                _align[0] = torch.zeros(1, dtype=torch.int32, device=dev)
            dist.all_reduce(_align[0])

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    nch = args.chunks
    nsamp = nch * 32768
    pl = build_plan(FS, 'h', DEC, [CENTER], correct_iq=True, demod='fm', omega_out=OMEGA)
    # the product's multi-GPU driver (sdrterm_b200/multigpu.py): one contiguous time segment per rank,
    # IQ-corrector state handed off on the device (no host round trip)
    chain = multigpu.TimeShardedChain(pl, nch, local, dist if world > 1 else None, torch)
    eng = chain.engine
    raw = synth_c1_device(torch, nsamp, seed=5 + rank, device=dev)
    out = torch.empty((1, nch * pl.M), dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        chain.step(raw.data_ptr(), nch, out.data_ptr(), stream)

    # ---------------- verify: the sharded result equals one pass over the concatenated stream
    verify = None
    if not args.no_verify:
        vch = min(nch, args.verify_chunks)
        chain.step(raw.data_ptr(), vch, out.data_ptr(), stream)
        torch.cuda.synchronize()
        mine = out[:, :vch * pl.M].clone()
        if world > 1:
            allraw = [torch.empty(vch * CB, dtype=torch.uint8, device=dev) for _ in range(world)]
            dist.all_gather(allraw, raw[:vch * CB].contiguous())
            allout = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allout, mine)
        else:
            allraw, allout = [raw[:vch * CB]], [mine]
        if rank == 0:
            whole = torch.cat(allraw)
            with Engine(pl, max_chunks=world * vch, device=local) as one:
                ref = torch.empty((1, world * vch * pl.M), dtype=torch.float64, device=dev)
                one.process_device(whole.data_ptr(), world * vch, ref.data_ptr(), stream)
                torch.cuda.synchronize()
            got = torch.cat(allout, dim=1)
            err = float((got - ref).abs().max() / ref.abs().max())
            verify = {'time_sharded_vs_single_pass': err, 'chunks_per_rank': vch, 'tolerance': 1e-9,
                      'note': 'the single pass itself is checked against the CPU oracle by tests/ (-m gpu) and smoke()'}

    clocks = Clocks(local)
    eng.set_profiling(world == 1)
    if rank == 0:
        clocks.start()                      # nvidia-smi needs ~0.1 s to produce its first row
    # the same step, untimed, for >= 0.3 s: brings the clocks under load before the timed region
    # (every rank runs the SAME number of steps: with N > 1 a step contains a collective)
    torch.cuda.synchronize()
    t_pre = time.perf_counter()
    step_device()
    torch.cuda.synchronize()
    t_one = max(time.perf_counter() - t_pre, 1e-4)
    extra = int(min(2000, 0.3 / t_one))
    if world > 1:
        tt = torch.tensor([extra], dtype=torch.int64, device=dev)
        dist.broadcast(tt, src=0)
        extra = int(tt.item())
    for i in range(args.warmup + extra):
        step_device()
        if i % 16 == 15:
            torch.cuda.synchronize()
    barrier()
    if world == 1:
        # one GPU carries the IQ corrector's offset from step to step, and how many steps ran above
        # depends on timing: the timed steps start from a zero offset, so what they compute depends
        # on the arguments only
        eng.iq_state = 0j
    l0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ktimes = []
    align_on_device()
    ev0.record()
    for _ in range(args.steps):
        step_device()
        if world == 1:
            ktimes.append(None)   # read after the loop's final sync for the last step only
    ev1.record()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = eng.launches - l0
    dumped = None
    if args.dump_outputs:
        dumped = out.clone()                # the steps below overwrite `out`
        if world > 1:
            parts = [torch.empty_like(dumped) for _ in range(world)]
            dist.all_gather(parts, dumped)
            dumped = torch.cat(parts, dim=1)
        dumped = dumped.cpu().numpy() if rank == 0 else None
    kt = eng.kernel_times() if world == 1 else None
    # a few extra profiled steps for a steadier per-kernel average
    kavg = None
    if world == 1:
        acc = np.zeros(4)
        reps = max(3, args.steps)
        for _ in range(reps):
            step_device()
            torch.cuda.synchronize()
            acc += np.array(eng.kernel_times())
        kavg = (acc / reps).tolist()
    # keep the identical step running so that the sampler sees it for ~0.3 s more (same count on
    # every rank)
    for i in range(extra):
        step_device()
        if i % 16 == 15:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    if rank == 0:
        clocks.stop()
    ms_step = ms_total / args.steps
    value = world * nsamp / (ms_step * 1e-3) / 1e6

    # ---------------- e2e: host pinned buffers through sdrb_submit / sdrb_wait
    sub = min(args.e2e_batch, nch)
    e2e_ch = min(nch, args.e2e_chunks)
    e2e_val = None
    if e2e_ch > 0:
        e2e_val = measure_e2e(torch, Engine, pl, raw, sub, e2e_ch, local, args, barrier, max_over_ranks, world)
    cli = None
    if world == 1 and args.cli_chunks > 0:
        cli = measure_cli(torch, raw, max(64, args.cli_chunks // 8), args.cli_chunks)
    # ---------------- SIMO banks (configs 3 and 4): sdrterm_b200.multigpu.RowShardedBank
    import signals

    def run_bank(label, fs, enc, rows_all, synth, sch, nsamp_chunk, steps, **plan_kw):
        bank = multigpu.RowShardedBank(fs, enc, 64, rows_all, sch, local, dist if world > 1 else None, torch,
                                       demod='fm', **plan_kw)
        cbk = bank.chunk_bytes
        leader = bank.rank == bank.leader
        raws = synth(bank.tg) if leader else torch.empty(sch * cbk, dtype=torch.uint8, device=dev)
        outs = torch.empty((len(bank.rows), sch * bank.M), dtype=torch.float64, device=dev)
        # ---- verify: this rank's rows of its segment == the same rows of a one-GPU pass over the
        #      whole bank on the segment's bytes (run by the group's leader)
        ver = None
        if not args.no_verify:
            vch = min(sch, 16)
            bank.run([raws[:vch * cbk]], vch, [outs], stream)
            torch.cuda.synchronize()
            mine = outs.reshape(-1)[:len(bank.rows) * vch * bank.M].reshape(len(bank.rows), vch * bank.M).clone()
            full_err = torch.zeros(1, dtype=torch.float64, device=dev)
            if bank.row_groups > 1:
                nmax = -(-len(rows_all) // bank.row_groups)
                pad = torch.zeros((nmax, vch * bank.M), dtype=torch.float64, device=dev)
                pad[:len(bank.rows)] = mine
                parts = [torch.empty_like(pad) for _ in range(bank.row_groups)]
                dist.all_gather(parts, pad, group=bank.group)
            else:
                parts = [mine]
            if leader:
                plf = build_plan(fs, enc, 64, rows_all, simo=True, demod='fm', **plan_kw)
                with Engine(plf, max_chunks=vch, device=local) as one:
                    ref = torch.empty((len(rows_all), vch * plf.M), dtype=torch.float64, device=dev)
                    one.process_device(raws.data_ptr(), vch, ref.data_ptr(), stream)
                    torch.cuda.synchronize()
                from sdrterm_b200 import sharding as shd
                got = torch.cat([parts[g][:shd.row_shard(len(rows_all), bank.row_groups, g)[1]
                                          - shd.row_shard(len(rows_all), bank.row_groups, g)[0]]
                                 for g in range(bank.row_groups)])
                # framed big-endian: compare the byte patterns' numeric values
                a = got.view(torch.uint8).reshape(-1, 8).flip(1).contiguous().view(torch.float64)
                b = ref.view(torch.uint8).reshape(-1, 8).flip(1).contiguous().view(torch.float64)
                full_err[0] = (a - b).abs().max() / b.abs().max()
            if world > 1:
                dist.all_reduce(full_err, op=dist.ReduceOp.MAX)
            ver = float(full_err.item())
        batches = [raws] * steps

        def go(n):
            bank.run(batches[:n], sch, [outs] * n, stream)

        go(3)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        align_on_device()
        e0.record()
        tc0 = time.perf_counter()
        go(steps)
        host_ms = (time.perf_counter() - tc0) * 1e3 / steps      # host time to enqueue one batch (not a rate)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        host_ms = max_over_ranks(host_ms)
        in_msps = bank.time_groups * sch * nsamp_chunk / (ms * 1e-3) / 1e6
        isz2 = cbk // nsamp_chunk
        bps = isz2 + 8 * len(rows_all) / 64
        res = {'workload': label, 'rows': len(rows_all), 'grid': {'row_groups': bank.row_groups, 'time_groups': bank.time_groups},
               'raw_transport': bank.transport, 'host_enqueue_ms_per_step': host_ms,
               'rows_on_rank0': len(bank.rows), 'chunks_per_step_per_time_group': sch,
               'input_msps': in_msps, 'vfo_msps': in_msps * len(rows_all), 'ms_per_step': ms, 'bytes_per_sample': bps,
               'front_end': 'k_tc' if bank.engine.tc is not None else 'k_main', 'verified_max_rel_err': ver}
        bank.close()
        return res

    simo = simo4 = None
    if args.simo_chunks > 0:
        offs = signals.vfo_grid(16, 100_000)
        simo = run_bank('config 3: 16 VFOs + centre (17 rows), int16 big-endian IQ, fs 2.4 MS/s, FM, -d 64; ranks on a '
                        '(row group x time group) grid, the raw batch of a time group sent to its ranks inside the '
                        'timed region (NVLink peer copies or ncclBroadcast, see raw_transport; pipelined against the kernels)',
                        2_400_000, 'h', [o for o in offs] + [0],
                        lambda tg: synth_c3_device(torch, args.simo_chunks * 32768, 3 + tg, dev, offs),
                        args.simo_chunks, 32768, 24, swap=True, omega_out=5000)
    if args.simo4_chunks > 0:
        offs4 = signals.vfo_grid(256, 200_000)

        def synth4(tg):
            g = torch.Generator(device=dev)
            g.manual_seed(4 + tg)
            n = args.simo4_chunks * 16384
            z = 0.05 * torch.randn((n, 2), generator=g, device=dev, dtype=torch.float32)
            t = torch.arange(n, device=dev, dtype=torch.float64) / 61_440_000
            for i in (0, 37, 128, 200, 255):         # a few of the 257 carriers (the rate does not depend on the signal)
                ph = 2 * torch.pi * offs4[i] * t + 0.11 * i
                z[:, 0] += (0.2 * torch.cos(ph)).float()
                z[:, 1] += (0.2 * torch.sin(ph)).float()
            return z.view(torch.uint8).reshape(-1)

        simo4 = run_bank('config 4: 256 VFOs + centre (257 rows) on 61.44 MS/s float32 IQ, FM, -d 64; rows sharded '
                         'over the ranks, every raw batch sent to all of them inside the timed region (raw_transport)',
                         61_440_000, 'f', [o for o in offs4] + [0], synth4, args.simo4_chunks, 16384, 12,
                         omega_out=12500)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if dumped is not None:
        write_outputs(args.dump_outputs, {'out': dumped})

    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak = json.load(open(peaks_path))['hbm_gbs']
        peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs, burst copy)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    bytes_per_sample = 4 + 8 * 1 / 64
    roof = None
    if kavg is not None:
        ach = bytes_per_sample * nsamp / (kavg[0] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tpath):
            try:
                per_chunk = json.load(open(tpath)).get('k_tc_dram_bytes_per_chunk')
                traffic = per_chunk * nch if (per_chunk and eng.tc is not None) else None
            except Exception:
                traffic = None
        kname = 'k_tc' if eng.tc is not None else 'k_main'
        roof = {'bound': 'hbm', 'kernel': kname, 'achieved': ach, 'peak': peak, 'unit': 'GB/s',
                'frac': ach / peak, 'traffic': traffic, 'peak_source': peak_src,
                'algorithmic_bytes_per_sample': bytes_per_sample,
                'kernel_ms': {kname: kavg[0], 'k_iqgain+k_iqscan+k_iqtiles': kavg[1],
                              'k_finish (or k_fixup)': kavg[2], 'k_demod (general path only)': kavg[3]},
                'algorithmic_bytes_per_launch': bytes_per_sample * nsamp,
                'traffic_source': 'profiles/traffic.json: ncu dram bytes per chunk x chunks per launch',
                'note': 'dominant kernel = block front end; k_tc = tcgen05 int8 GEMM over the raw bytes + FP64 epilogue (DESIGN.md 3.4)'}
        for sm in (simo, simo4):
            if sm is not None:
                sm['frac_hbm'] = sm['input_msps'] * 1e6 * sm['bytes_per_sample'] / 1e9 / peak / world
    cpu = None
    if world == 1 and not args.no_cpu:
        nth = host_threads()
        v, sample = cpu_chain_rate(64, args.cpu_seconds, nth)
        cpu = {'value': v, 'unit': 'Msamples/s', 'cores': nth, 'kind': 'port', 'sample': sample}
    line = {'metric': METRIC, 'value': value, 'unit': 'Msamples/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'chunks_per_gpu_per_step': nch,
                       'l2': 'inputs larger than L2 (1 GiB per step per GPU)',
                       'parallelism': 'time-segment sharding, IQ state via all-gather' if world > 1 else 'single GPU'},
            'e2e': None if e2e_val is None else {'value': e2e_val, 'unit': 'Msamples/s', 'h2d_bytes_per_step': e2e_ch * CB,
                    'd2h_bytes_per_step': e2e_ch * pl.M * 8,
                    'note': f'{e2e_ch} chunks per step in batches of {sub}, double-buffered sdrb_submit/sdrb_wait',
                    'numa_bound': numa_bound, 'cpus_after_binding': numa_cpus},
            'gpu_launches': launches, 'clocks': clocks.summary()}
    if roof is not None:
        line['roofline'] = roof
    if cpu is not None:
        line['cpu_baseline'] = cpu
    if cli is not None:
        line['cli_e2e'] = cli
    if simo is not None:
        line['simo'] = simo
    if simo4 is not None:
        line['simo_config4'] = simo4
    if verify is not None:
        errs = [verify['time_sharded_vs_single_pass']]
        errs += [sm['verified_max_rel_err'] for sm in (simo, simo4) if sm is not None and sm['verified_max_rel_err'] is not None]
        line['verify'] = verify
        line['verified'] = bool(all(e == e and e <= 1e-9 for e in errs))
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None
_ALL_CPUS = None


def claim_stdout():
    """Keep the real stdout for the one JSON line: everything else written to fd 1 from here on
    (NCCL prints its version banner and its NCCL_DEBUG output there) goes to stderr instead, so no
    NCCL_DEBUG override is needed to keep the line parseable."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + '\n').encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_BYTES = 64_000_000


def write_outputs(d: str, arrays: dict) -> None:
    """Save each array as d/<name>.npy in float64.  Past DUMP_BYTES in all, an array keeps the same
    seeded sample of its last axis at every run with the same shapes."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    budget = (DUMP_BYTES - 4096 * len(arrays)) // len(arrays)          # 4096: room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > budget:
            keep = budget // (8 * (a.size // a.shape[-1]))
            cols = np.sort(np.random.default_rng(0).choice(a.shape[-1], keep, replace=False))
            a = a[..., cols]
        np.save(os.path.join(d, name + '.npy'), np.ascontiguousarray(a))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5,
                    help='timed steps of the headline measurement (the e2e and SIMO legs keep their own counts)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--chunks', type=int, default=8192, help='chunks per GPU per step')
    ap.add_argument('--e2e-chunks', type=int, default=4096)
    ap.add_argument('--e2e-batch', type=int, default=512)
    ap.add_argument('--simo-chunks', type=int, default=512)
    ap.add_argument('--simo4-chunks', type=int, default=256, help='config 4 (257 rows, float32) chunks per step')
    ap.add_argument('--cli-chunks', type=int, default=8192, help='chunks of the larger file of the CLI end-to-end leg (0 = skip)')
    ap.add_argument('--no-numa', action='store_true', help='do not bind the rank to its GPU\'s NUMA node')
    ap.add_argument('--no-verify', action='store_true', help='skip the output verification legs')
    ap.add_argument('--verify-chunks', type=int, default=64)
    ap.add_argument('--ref-chunks', type=int, default=1024, help='chunks per step of the reference arm')
    ap.add_argument('--cpu-seconds', type=float, default=10.0)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the last timed step\'s output to DIR/out.npy (float64, at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    claim_stdout()
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_cuda_arm(args)


if __name__ == '__main__':
    main()
