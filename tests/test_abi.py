"""C-ABI surface (no GPU needed): the library builds for sm_100a, loads, and exports every function
include/sdrterm_b200.h declares; the ctypes structures match the header's layout-relevant constants;
compute entry points fail loudly (never fall back) without a CUDA device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from sdrterm_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'sdrterm_b200.h')


def _declared():
    src = open(HEADER).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(sdrb_[a-z_0-9]+)\s*\(', src)))


def test_library_builds_and_exports_every_declared_symbol():
    path = nat.build()
    assert os.path.exists(path)
    lib = C.CDLL(path)
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f'{n} declared in the header but not exported'
    assert set(nat.EXPORTS) <= set(names)
    assert set(names) == set(nat.EXPORTS), set(names) ^ set(nat.EXPORTS)


def test_every_csrc_file_is_a_rebuild_dependency():
    """build() recompiles when a file in SOURCES is newer than the library: a header left out would
    let an edit to it run against the stale library."""
    csrc = os.path.join(ROOT, 'sdrterm_b200', 'csrc')
    assert sorted(os.path.join(csrc, f) for f in os.listdir(csrc)) == sorted(nat.SOURCES)


def test_abi_version_matches_header():
    m = re.search(r'#define SDRB_ABI_VERSION (\d+)', open(HEADER).read())
    assert int(m.group(1)) == nat.ABI_VERSION


def test_build_targets_sm_100a_only():
    cmd = ' '.join(nat.nvcc_command())
    assert 'arch=compute_100a,code=sm_100a' in cmd and '-lineinfo' in cmd
    sass = os.popen(f'cuobjdump -lelf {nat.LIB_PATH} 2>/dev/null').read()
    assert 'sm_100a' in sass and 'sm_90' not in sass


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry point reports an error; nothing computes on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    from sdrterm_b200.engine import Engine
    from sdrterm_b200.plan import build_plan
    pl = build_plan(1_024_000, 'h', 64, [15000], correct_iq=True, demod='fm', omega_out=5000)
    with pytest.raises(nat.SdrbError, match='no CUDA device'):
        Engine(pl, max_chunks=1)
    import sdrterm_b200.dsp.demodulation as dem
    with pytest.raises(nat.SdrbError):
        dem.amDemod(np.zeros((1, 8), dtype=np.complex128), np.zeros((1, 8)))


def test_create_refuses_inconsistent_plans_before_touching_the_device():
    """sdrb_create checks the whole configuration on the host before any CUDA call: an inconsistent
    plan is refused with SDRB_ERR_ARG naming the problem, with or without a CUDA device."""
    import dataclasses
    from sdrterm_b200.engine import Engine
    from sdrterm_b200.plan import build_plan
    kw = dict(correct_iq=True, demod='fm', omega_out=5000)
    fm = build_plan(1_024_000, 'h', 64, [15000], **kw)
    fm_d50 = build_plan(1_024_000, 'h', 50, [15000], **kw)        # M = 656: FM needs the dense interpolation
    seamless = build_plan(1_024_000, 'h', 64, [15000], seamless=True, **kw)
    assert fm_d50.fm_interp is not None and seamless.lookahead >= 1
    for pl, problem in ((dataclasses.replace(fm, RL=fm.RL + 1), 'RL'),
                        (dataclasses.replace(fm_d50, fm_interp=None), 'dense interpolation table'),
                        (dataclasses.replace(seamless, lookahead=0), 'lookahead'),
                        (dataclasses.replace(fm, edge=32), 'filter pad 32')):     # the head is one warp of samples
        with pytest.raises(nat.SdrbError, match=f'error -1: .*{problem}'):
            Engine(pl, max_chunks=1, use_tc=False)


def test_product_code_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'sdrterm_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert 'oracle' not in src.replace('the oracle', '').replace("oracle's", ''), os.path.join(dirpath, f)
