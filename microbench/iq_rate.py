"""Device-resident cost of the complex baseband output (-m iq) against fm, 1 GiB of raw input per
step (larger than L2), CUDA events, warm-ups, the modes alternating in one run:

  * config 1 (int16 IQ at 1.024 MS/s, -d 64, --correct-iq, centre 15 kHz), default chain: fm vs iq,
    with the k_finish share from the handle's kernel timers;
  * the same in seamless mode: fm vs iq;
  * config 3's 17-row bank (int16 big-endian at 2.4 MS/s, 16 VFOs + centre, -d 64): fm vs iq.

Algorithmic bytes per input sample for config 1: 4 in, plus per output (one per 64 samples) 8 for fm,
16 for iq: 4.125 vs 4.25 B/sample.  The card's name and power limit are read in the same run.  Writes
profiles/iq_rate.json (or the directory given as argv[1])."""
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
    res['ratio_iq_over_fm'] = res['step_ms']['iq'] / res['step_ms']['fm']
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
    print(label, json.dumps(res['step_ms']), f"iq/fm = {res['ratio_iq_over_fm']:.3f}", flush=True)
    return res


def main(outdir):
    st = torch.cuda.current_stream().cuda_stream
    res = {'card': card(), 'raw_bytes_per_step': NCH * 131072}
    raw = torch.randint(-2000, 2000, (NCH * 65536,), dtype=torch.int16, device='cuda').view(torch.uint8)
    for seamless in (False, True):
        label = 'config1_seamless' if seamless else 'config1_default'
        engines = {d: Engine(build_plan(1_024_000, 'h', 64, [15000], correct_iq=True, demod=d, omega_out=5000,
                                        seamless=seamless), max_chunks=NCH) for d in ('fm', 'iq')}
        res[label] = compare(label, engines, raw, st)
        for e in engines.values():
            e.close()
    vfos = [k * 100_000 for k in range(-8, 0)] + [k * 100_000 for k in range(1, 9)]
    engines = {d: Engine(build_plan(2_400_000, 'h', 64, vfos + [0], simo=True, swap=True, demod=d, omega_out=5000),
                         max_chunks=NCH) for d in ('fm', 'iq')}
    res['config3_bank17'] = compare('config3_bank17', engines, raw, st)
    for e in engines.values():
        e.close()
    res['config1'] = 'int16 -d 64 --correct-iq, 1.024 MS/s, centre 15 kHz, 2^28 samples per step'
    res['config3'] = 'int16 big-endian, 2.4 MS/s, 16 VFOs on a 100 kHz grid + centre, -d 64, 2^28 samples per step'
    res['algorithmic_bytes_per_sample_config1'] = {'fm': 4 + 8 / 64, 'iq': 4 + 16 / 64}
    for label in ('config1_default', 'config1_seamless'):
        res[label]['input_Msamples_per_s'] = {k: NCH * 32768 / (v * 1e3) for k, v in res[label]['step_ms'].items()}
    print(json.dumps(res, indent=1))
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, 'iq_rate.json'), 'w') as fh:
        json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles'))
