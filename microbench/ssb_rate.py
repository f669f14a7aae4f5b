"""Device-resident cost of single-sideband output (-m usb, -w 3000) against fm (-w 5000), 1 GiB of raw
input per step (larger than L2), CUDA events, warm-ups, the modes alternating in one run:

  * config 1 (int16 IQ at 1.024 MS/s, -d 64, --correct-iq, centre 15 kHz), default chain: fm vs usb,
    with the kernel-group shares from the handle's timers;
  * the same in seamless mode: fm vs usb;
  * config 3's 17-row bank (int16 big-endian at 2.4 MS/s, 16 VFOs + centre, -d 64): fm vs usb.

Then, in a separate pass, torch.profiler gives the per-kernel device time of one step of every
workload and mode (k_finish, k_fixup / k_demod, k_seam_*).  Both modes write 8 bytes per output.  The
card's name and power limit are read in the same run.  Writes profiles/ssb_rate.json (or the
directory given as argv[1])."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
import torch  # noqa: E402

from sdrterm_b200.engine import Engine  # noqa: E402
from sdrterm_b200.plan import build_plan  # noqa: E402

NCH = 8192                 # 8192 chunks x 131072 bytes = 1 GiB of raw input per step
REPS, ROUNDS, WARM = 5, 4, 3


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def _step(eng, raw, out, st):
    if eng.seamless:
        return lambda: eng.stream_device(raw.data_ptr(), NCH, out.data_ptr(), st)
    return lambda: eng.process_device(raw.data_ptr(), NCH, out.data_ptr(), st)


def compare(label, engines, raw, st):
    """Alternate the modes of one workload; min over rounds of the mean of REPS steps."""
    W = max(e.R * e.W for e in engines.values())
    out = torch.empty((NCH * W,), dtype=torch.float64, device='cuda')
    steps = {name: _step(e, raw, out, st) for name, e in engines.items()}
    for f in steps.values():
        for _ in range(WARM):
            f()
    torch.cuda.synchronize()
    times = {name: [] for name in steps}
    for _ in range(ROUNDS):
        for name, f in steps.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(REPS):
                f()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / REPS)
    res = {'step_ms': {k: min(v) for k, v in times.items()}, 'step_ms_all_rounds': times}
    res['ratio_usb_over_fm'] = res['step_ms']['usb'] / res['step_ms']['fm']
    for name, e in engines.items():
        if not e.seamless:                   # kernel groups of one more step: front end | IQ | finish | demod
            e.set_profiling(True)
            steps[name]()
            torch.cuda.synchronize()
            res.setdefault('kernel_ms', {})[name] = [round(v, 4) for v in e.kernel_times()]
            e.set_profiling(False)
        else:
            e.stream_end_device(out.data_ptr(), st)
    torch.cuda.synchronize()
    res['kernel_us_per_step'] = {name: profile(e, steps[name], out, st) for name, e in engines.items()}
    print(label, json.dumps(res['step_ms']), f"usb/fm = {res['ratio_usb_over_fm']:.3f}", flush=True)
    return res


def profile(eng, step, out, st, n=3):
    """Device time per step and kernel (microseconds) over n steps, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile as prof
    with prof(activities=[ProfilerActivity.CUDA]) as p:
        for _ in range(n):
            step()
        torch.cuda.synchronize()
    if eng.seamless:
        eng.stream_end_device(out.data_ptr(), st)
        torch.cuda.synchronize()
    acc = {}
    for ev in p.key_averages():
        t = getattr(ev, 'device_time_total', None)
        if t is None:
            t = ev.cuda_time_total
        name = ev.key.split('(')[0]
        name = name[5:] if name.startswith('void ') else name
        if t > 0 and name.startswith('k_'):
            acc[name] = acc.get(name, 0.0) + t / n
    return {k: round(v, 2) for k, v in sorted(acc.items(), key=lambda kv: -kv[1])}


MODES = {'fm': 5000, 'usb': 3000}     # -w: fm's output low-pass, usb's sideband width


def main(outdir):
    st = torch.cuda.current_stream().cuda_stream
    res = {'card': card(), 'raw_bytes_per_step': NCH * 131072}
    raw = torch.randint(-2000, 2000, (NCH * 65536,), dtype=torch.int16, device='cuda').view(torch.uint8)
    for seamless in (False, True):
        label = 'config1_seamless' if seamless else 'config1_default'
        engines = {d: Engine(build_plan(1_024_000, 'h', 64, [15000], correct_iq=True, demod=d, omega_out=w,
                                        seamless=seamless), max_chunks=NCH) for d, w in MODES.items()}
        res[label] = compare(label, engines, raw, st)
        for e in engines.values():
            e.close()
    vfos = [k * 100_000 for k in range(-8, 0)] + [k * 100_000 for k in range(1, 9)]
    engines = {d: Engine(build_plan(2_400_000, 'h', 64, vfos + [0], simo=True, swap=True, demod=d, omega_out=w),
                         max_chunks=NCH) for d, w in MODES.items()}
    res['config3_bank17'] = compare('config3_bank17', engines, raw, st)
    for e in engines.values():
        e.close()
    res['config1'] = 'int16 -d 64 --correct-iq, 1.024 MS/s, centre 15 kHz, 2^28 samples per step'
    res['config3'] = 'int16 big-endian, 2.4 MS/s, 16 VFOs on a 100 kHz grid + centre, -d 64, 2^28 samples per step'
    res['algorithmic_bytes_per_sample_config1'] = {'fm': 4 + 8 / 64, 'usb': 4 + 8 / 64}
    for label in ('config1_default', 'config1_seamless'):
        res[label]['input_Msamples_per_s'] = {k: NCH * 32768 / (v * 1e3) for k, v in res[label]['step_ms'].items()}
    print(json.dumps(res, indent=1))
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, 'ssb_rate.json'), 'w') as fh:
        json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles'))
