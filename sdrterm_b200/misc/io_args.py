"""``IOArgs``: the wiring object of the reference's CLI (src/misc/io_args.py:27-141): picks the
processor class (``DspProcessor`` / ``VfoProcessor`` for ``--simo``), selects the demodulation and
wraps ``processor.processData`` in a ``multiprocessing.Process`` fed by a fresh ``Queue`` -- the
processor pickles into a spawned child without CUDA state and builds its engine there.  Plot
consumers are out of scope of this build (DESIGN.md 9): ``selectPlotType`` reports that and returns
None, exactly what the reference does when pyqtgraph is missing."""
from __future__ import annotations

from enum import Enum
from multiprocessing import Process, Queue
from typing import Callable

from .general_util import eprint, tprint, traceOn, verboseOn


class DemodulationChoices(str, Enum):
    FM = 'fm'
    AM = 'am'
    REAL = 're'
    IMAG = 'im'
    IQ = 'iq'
    USB = 'usb'
    LSB = 'lsb'

    def __str__(self):
        return self.value


def selectDemodulation(demodType, processor) -> Callable:
    tprint(f'{demodType} requested')
    table = {'fm': 'selectOutputFm', 'nfm': 'selectOutputFm', 'am': 'selectOutputAm',
             're': 'selectOutputReal', 'im': 'selectOutputImag', 'iq': 'selectOutputIq',
             'usb': 'selectOutputUsb', 'lsb': 'selectOutputLsb'}
    name = table.get(str(demodType.value if isinstance(demodType, Enum) else demodType))
    if name is None:
        raise ValueError(f'Invalid demod type {demodType}')
    return getattr(processor, name)


def selectPlotType(plotType):
    from importlib.util import find_spec
    if find_spec('pyqtgraph') is None:
        eprint('pyqtgraph not installed')
        return None
    if str(plotType) in ('ps', 'spec', 'vfos', 'vfo', 'water', 'waterfall'):
        eprint('plots are not part of the B200 build')
        return None
    raise ValueError(f'Invalid plot type {plotType}')


class IOArgs:
    strct = None

    def __init__(self, verbose: int = 0, **kwargs):
        from .file_util import checkWavHeader
        IOArgs.strct = kwargs
        if verbose > 1:
            traceOn()
        elif verbose > 0:
            verboseOn()
        kwargs['fileInfo'] = checkWavHeader(kwargs['inFile'], kwargs['fs'], kwargs['enc'])
        kwargs['fs'] = kwargs['fileInfo']['sampRate']
        IOArgs._initializeOutputHandlers(**kwargs)
        kwargs['isDead'].value = 0

    @classmethod
    def _initializeProcess(cls, isDead, processor, *args, name: str = 'Process', **kwargs):
        if processor is None:
            raise ValueError('Processor must be provided')
        buffer = Queue()
        proc = Process(target=processor.processData, args=(isDead, buffer, *args), kwargs=kwargs)
        proc.name = name + str(processor)
        return buffer, proc

    @classmethod
    def _initializeOutputHandlers(cls, isDead=None, fs: int = 0, dm=None, outFile: str | None = None,
                                  simo: bool = False, pl: str | None = None, processes: list | None = None,
                                  buffers: list | None = None, **kwargs) -> None:
        if simo:
            from ..dsp.vfo_processor import VfoProcessor as Processor
        else:
            from ..dsp.dsp_processor import DspProcessor as Processor
        cls.strct['processor'] = Processor(fs, **kwargs)
        selectDemodulation(dm, cls.strct['processor'])()
        if pl:
            for p in pl.split(','):
                selectPlotType(p)                     # reports; plot consumers are not built
        buffer, proc = cls._initializeProcess(isDead, cls.strct['processor'], outFile, name='File writer-', **kwargs)
        processes.append(proc)
        buffers.append(buffer)
