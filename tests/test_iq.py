"""Complex baseband output (``-m iq``) without a GPU: the plan, the oracle, the golden vectors, the
C-ABI constant and the host layers (CLI, processors)."""
import os
import pickle
import re

import numpy as np
import pytest

from iq_ref import interleave, iq_oracle
from oracle import oracle as orc
from sdrterm_b200 import _native as nat
from sdrterm_b200.plan import build_plan
from util import case_stream, load_golden, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plan_iq_has_no_output_filter_and_two_doubles_per_output():
    pl = build_plan(1_024_000, 'h', 64, [15000], correct_iq=True, demod='iq', omega_out=5000)
    assert pl.out_sos is None and pl.sos_AL is None and pl.fm_interp is None
    assert pl.M == 512 and pl.W == 2 * pl.M
    assert nat.DEMOD_CODE[pl.demod] == nat.IQ == 4
    for demod in ('fm', 'am', 're', 'im'):
        assert build_plan(1_024_000, 'h', 64, [15000], demod=demod, omega_out=5000).W == 512
    ragged = build_plan(2_400_000, 'B', 50, [0], demod='iq')
    assert ragged.M == 1311 and ragged.W == 2622


def test_oracle_iq_is_interleaved_re_and_im():
    raw, body, kw = case_stream('c1_fm_wav_int16')
    out = iq_oracle(kw, body)
    re_ = orc.Chain(**{**kw, 'demod': 're'}).run(body)
    im_ = orc.Chain(**{**kw, 'demod': 'im'}).run(body)
    assert out.shape == (1, 2 * re_.shape[1])
    assert np.array_equal(out, interleave(re_, im_))
    assert np.array_equal(out[:, 0::2], re_) and np.array_equal(out[:, 1::2], im_)


@pytest.mark.parametrize('name,col', [('enc_b_re', 0), ('enc_H_swap_im', 1)])
def test_oracle_iq_columns_match_reference_golden(name, col):
    """The real column against the reference's own `-m re` output, the imaginary column against
    its `-m im` output, each on that golden's case."""
    raw, body, kw = case_stream(name)
    g = load_golden(name)
    out = iq_oracle(kw, body)
    assert out[:, col::2].shape == g['out'].shape
    assert rel_err(out[:, col::2], g['out']) < 2e-11


def test_header_iq_constant_matches_python():
    src = open(os.path.join(ROOT, 'include', 'sdrterm_b200.h')).read()
    m = re.search(r'enum sdrb_demod \{([^}]*)\}', src)
    consts = dict((k, int(v)) for k, v in re.findall(r'(SDRB_\w+) = (\d+)', m.group(1)))
    assert consts['SDRB_IQ'] == nat.IQ == nat.DEMOD_CODE['iq']


def test_cli_parser_accepts_iq():
    from sdrterm_b200.dsp import demodulation as dem
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    from sdrterm_b200.dsp.vfo_processor import VfoProcessor
    from sdrterm_b200.misc import file_util
    from sdrterm_b200.misc.io_args import DemodulationChoices, selectDemodulation
    from sdrterm_b200.sdrterm import buildParser, makeProcessor
    a = buildParser().parse_args(['-r', '1024k', '-c', '15k', '-d', '64', '-e', 'h', '-m', 'IQ'])
    assert a.demod == 'iq'
    p = makeProcessor(a, file_util.parseRawType(None, a.fs, a.enc))
    assert isinstance(p, DspProcessor) and p.demod == dem.iqOutput and p.bandwidth == p.decimatedFs == 16000
    b = buildParser().parse_args(['-r', '2400k', '-e', 'h', '--simo', '--vfos', '100000', '-d', '64', '-m', 'iq',
                                  '--vfo-host', '127.0.0.1:0'])
    v = makeProcessor(b, file_util.parseRawType(None, b.fs, b.enc))
    assert isinstance(v, VfoProcessor) and v.demod == dem.iqOutput and v._demodName() == 'iq'
    assert str(DemodulationChoices.IQ) == 'iq'
    q = DspProcessor(48000)
    selectDemodulation(DemodulationChoices.IQ, q)()
    assert q.demod == dem.iqOutput


def test_select_output_iq_and_pickle_keep_the_mode():
    from sdrterm_b200.dsp import demodulation as dem
    from sdrterm_b200.dsp.dsp_processor import DspProcessor
    p = DspProcessor(1_024_000, center=15000, omegaOut=5000, dec=64, enc='h', correctIq=True)
    p.selectOutputIq()
    assert p.demod == dem.iqOutput and p._outputFilters == [] and p.bandwidth == p.decimatedFs
    assert p._demodName() == 'iq'
    q = pickle.loads(pickle.dumps(p))
    assert q.demod == dem.iqOutput and q._demodName() == 'iq' and q._engine is None


def test_iq_operator_checks_its_output_shape():
    from sdrterm_b200.dsp import demodulation as dem
    with pytest.raises(ValueError):
        dem.iqOutput(np.zeros((1, 8), dtype=np.complex128), np.zeros((1, 8)))


def test_cached_plan_keeps_modes_apart(tmp_path, monkeypatch):
    from sdrterm_b200.plan import cached_plan
    monkeypatch.setenv('SDRB_PLAN_CACHE', str(tmp_path))
    args = (2_400_000, 'f', 64, [30000])
    for demod in ('re', 'iq', 're'):
        pl, tc = cached_plan(*args, demod=demod, omega_out=5000)
        assert pl.demod == demod and pl.W == (2 if demod == 'iq' else 1) * pl.M
    assert len(list(tmp_path.glob('plan_*.pkl'))) == 2
