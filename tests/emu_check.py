"""Developer script: the numpy twins of the kernels vs the oracle for the parity cases
(python tests/emu_check.py [case ...]); tests/test_emulator.py runs a subset in the CPU suite."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
import numpy as np

from cases import CASES
from oracle import oracle as orc
from util import case_stream, load_golden, rel_err
from sdrterm_b200.plan import build_plan, build_tc
import emulator as emu

names = sys.argv[1:] or sorted(CASES)
for name in names:
    raw, body, kw = case_stream(name)
    g = load_golden(name)
    ch = orc.Chain(**kw)
    t = time.time()
    pl = build_plan(kw['fs'], kw['enc'], kw['dec'], ch.rows, simo=kw['simo'], swap=orc.needs_swap(ch.dt),
                    correct_iq=kw['correct_iq'], normalize=kw['normalize'], demod=kw['demod'], omega_out=kw['omega_out'])
    tp = time.time() - t
    out, ys, off = emu.emu_stream(pl, body)
    chunks = []
    ch2 = orc.Chain(**kw)
    for o in range(0, len(body), 131072):
        chunks.append(ch2.ingest(body[o:o + 131072]).copy())
    yo = ch2.decimated(np.stack(chunks))
    oo = orc.Chain(**kw).run(body)
    line = (f'{name:22s} plan {tp:5.2f}s  y vs oracle {rel_err(ys, yo):.2e}  out vs oracle {rel_err(out, oo):.2e}  '
            f'out vs ref {rel_err(out, g["out"]):.2e} off {abs(off - ch2._off[0]):.1e}')
    tc = build_tc(pl)
    if tc is not None:
        out2, ys2, off2 = emu.emu_stream_tc(pl, tc, body[:len(body) // 131072 * 131072] if len(body) % 131072 == 0 else body)
        line += f' | tc: y {rel_err(ys2, yo):.2e} out {rel_err(out2, oo):.2e}'
    print(line)
