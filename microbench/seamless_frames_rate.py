"""Device-resident cost of the seamless mode at a decimation that does not divide the chunk: BASELINE
config 2 (uint8 IQ at 2.4 MS/s, AM, -d 50 -w 5k, --correct-iq), 2^29 samples = 1 GiB of raw input per
step (larger than L2).  The default chain (sdrb_process_device, 8192 chunks of 65536 samples)
against the seamless mode fed through the sample entry (sdrb_stream_samples_device: frames of 64000
samples, the remainder carried on the device), CUDA events, warm-ups, the two modes alternating in
one run.  Then a torch.profiler pass of each mode for the per-kernel times, the device-to-device
copies of the sample entry included.  The card's name and power limit are read in the same run.
Writes profiles/seamless_frames_rate.json (or the directory given as argv[1])."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
import torch  # noqa: E402

from sdrterm_b200.engine import Engine  # noqa: E402
from sdrterm_b200.plan import build_plan, seamless_frame_samples  # noqa: E402

NCH = 8192                 # 8192 chunks x 65536 samples = 2^29 samples per step
NS = NCH * 65536
REPS, ROUNDS, WARM = 5, 4, 3


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def main(outdir):
    kw = dict(correct_iq=True, demod='am', omega_out=5000)
    nf = seamless_frame_samples(65536, 50)
    dflt = Engine(build_plan(2_400_000, 'B', 50, [0], **kw), max_chunks=NCH)
    seam = Engine(build_plan(2_400_000, 'B', 50, [0], seamless=True, chunk_bytes=2 * nf, **kw),
                  max_chunks=-(-NS // nf))
    raw = torch.randint(0, 256, (2 * NS,), dtype=torch.uint8, device='cuda')
    out = torch.empty((max(NCH * dflt.W, seam.stream_capacity(NS)),), dtype=torch.float64, device='cuda')
    st = torch.cuda.current_stream().cuda_stream

    def step_default():
        dflt.process_device(raw.data_ptr(), NCH, out.data_ptr(), st)

    def step_seamless():
        seam.stream_samples_device(raw.data_ptr(), NS, out.data_ptr(), st)

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
                k = 'memcpy ' + ev.name.split()[1] if len(ev.name.split()) > 1 else 'memcpy'
                agg[k] = agg.get(k, 0.0) + ev.device_time / 1e3 / 3
        kernels[name] = {k: round(v, 4) for k, v in sorted(agg.items(), key=lambda kv: -kv[1])}
    seam.stream_samples_end_device(out.data_ptr(), st)
    torch.cuda.synchronize()
    md, ms = min(times['default']), min(times['seamless'])
    res = {'card': card(), 'config': 'uint8 AM -d 50 -w 5k --correct-iq, 2.4 MS/s, centre 0 (BASELINE config 2)',
           'samples_per_step': NS, 'frame_samples': nf, 'step_ms': {'default': md, 'seamless': ms},
           'step_ms_all_rounds': times, 'ratio_seamless_over_default': ms / md,
           'lookahead': seam.lookahead, 'kernel_ms_per_step': kernels}
    print(json.dumps(res, indent=1))
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, 'seamless_frames_rate.json'), 'w') as fh:
        json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles'))
