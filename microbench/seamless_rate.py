"""Device-resident cost of the seamless streaming mode against the default chain, config 1
(int16 IQ at 1.024 MS/s, FM, -d 64, --correct-iq, centre 15 kHz), 2^28 samples per step (1 GiB of raw
input, larger than L2), CUDA events, warm-ups, the two modes alternating in one run.  Then a
torch.profiler pass of each mode for the per-kernel times.  The card's name and power limit are read
in the same run.  Writes profiles/seamless_rate.json (or the directory given as argv[1])."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
import torch  # noqa: E402

from sdrterm_b200.engine import Engine  # noqa: E402
from sdrterm_b200.plan import build_plan  # noqa: E402

NCH = 8192                 # 8192 chunks x 32768 samples = 2^28 samples per step
REPS, ROUNDS, WARM = 5, 4, 3


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def main(outdir):
    kw = dict(correct_iq=True, demod='fm', omega_out=5000)
    dflt = Engine(build_plan(1_024_000, 'h', 64, [15000], **kw), max_chunks=NCH)
    seam = Engine(build_plan(1_024_000, 'h', 64, [15000], seamless=True, **kw), max_chunks=NCH)
    raw = torch.randint(-2000, 2000, (NCH * 65536,), dtype=torch.int16, device='cuda').view(torch.uint8)
    out = torch.empty((NCH * seam.M,), dtype=torch.float64, device='cuda')
    st = torch.cuda.current_stream().cuda_stream

    def step_default():
        dflt.process_device(raw.data_ptr(), NCH, out.data_ptr(), st)

    def step_seamless():
        seam.stream_device(raw.data_ptr(), NCH, out.data_ptr(), st)

    for f in (step_default, step_seamless):
        for _ in range(WARM):
            f()
    torch.cuda.synchronize()
    times = {'default': [], 'seamless': []}
    for _ in range(ROUNDS):
        for name, f in (('default', step_default), ('seamless', step_seamless)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(REPS):
                f()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / REPS)
    kernels = {}
    from torch.profiler import ProfilerActivity, profile
    for name, f in (('default', step_default), ('seamless', step_seamless)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                f()
            torch.cuda.synchronize()
        agg = {}
        for ev in prof.events():
            if ev.device_type.name == 'CUDA' and ev.name.startswith(('k_', 'void k_')):
                k = ev.name.split('<')[0].replace('void ', '').split('(')[0]
                agg[k] = agg.get(k, 0.0) + ev.device_time / 1e3 / 3
            elif ev.device_type.name == 'CUDA' and 'Memcpy' in ev.name:
                agg['memcpy'] = agg.get('memcpy', 0.0) + ev.device_time / 1e3 / 3
        kernels[name] = {k: round(v, 4) for k, v in sorted(agg.items(), key=lambda kv: -kv[1])}
    seam.stream_end_device(out.data_ptr(), st)
    torch.cuda.synchronize()
    md, ms = min(times['default']), min(times['seamless'])
    res = {'card': card(), 'config': 'int16 FM -d 64 --correct-iq, 1.024 MS/s, centre 15 kHz',
           'samples_per_step': NCH * 32768, 'step_ms': {'default': md, 'seamless': ms},
           'step_ms_all_rounds': times, 'ratio_seamless_over_default': ms / md,
           'lookahead': seam.lookahead, 'kernel_ms_per_step': kernels}
    print(json.dumps(res, indent=1))
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, 'seamless_rate.json'), 'w') as fh:
        json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles'))
