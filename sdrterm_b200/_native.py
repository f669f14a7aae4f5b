"""ctypes binding of libsdrterm_b200.so (include/sdrterm_b200.h).

There is no CPU fallback: importing works anywhere (so the CPU test-suite can check that the
library loads and exports its symbols), but every compute entry point needs a CUDA device and
raises ``SdrbError`` otherwise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get('SDRB_LIB') or os.path.join(_HERE, 'libsdrterm_b200.so')   # SDRB_LIB: experiment builds
HEADER = os.path.join(ROOT, 'include', 'sdrterm_b200.h')
SOURCES = [os.path.join(_HERE, 'csrc', f) for f in ('sdrb_api.cu', 'sdrb_kernels.cuh', 'sdrb_device.cuh', 'sdrb_tc.cuh', 'sdrb_finish.cuh',
                                                    'sdrb_spectrum.cuh', 'sdrb_seamless.cuh', 'sdrb_outstage.cuh', 'sdrb_fft.cuh')]

ABI_VERSION = 11
FM, AM, RE, IM, IQ, USB, LSB = 0, 1, 2, 3, 4, 5, 6
DEMOD_CODE = {'fm': FM, 'am': AM, 're': RE, 'im': IM, 'iq': IQ, 'usb': USB, 'lsb': LSB}


class SdrbError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [('abi_version', C.c_int32), ('device', C.c_int32), ('enc', C.c_char),
                ('swap', C.c_uint8), ('correct_iq', C.c_uint8), ('normalize', C.c_uint8),
                ('demod', C.c_uint8), ('big_endian_out', C.c_uint8), ('seamless', C.c_uint8),
                ('reserved', C.c_uint8 * 1),
                ('q', C.c_int32), ('N', C.c_int32), ('edge', C.c_int32), ('R', C.c_int32),
                ('n_out_sections', C.c_int32), ('max_chunks', C.c_int32), ('iq_L', C.c_double),
                ('norm_xmin', C.c_double), ('norm_k', C.c_double)]


_DP = C.POINTER(C.c_double)


class Tables(C.Structure):
    _fields_ = [('p', _DP), ('P', _DP), ('rho', _DP), ('rho_p', _DP), ('c', _DP), ('zhat', _DP),
                ('xi', _DP), ('g0', C.c_double), ('d', C.c_double), ('Ec', _DP), ('Oc', _DP),
                ('Ppow', _DP), ('pk', _DP), ('Pt', _DP), ('bx', _DP), ('bnd', _DP), ('k_bnd', C.c_int32), ('lam', C.c_double),
                ('lam_q', C.c_double), ('lam_N', C.c_double), ('lam_inv', C.c_double),
                ('lam_j', _DP), ('lam_k', _DP), ('mu_k', _DP), ('lam_tile', C.c_double * 2), ('RL', C.c_int32),
                ('run_len', C.c_int32 * 8), ('lam_run', C.c_double * 8), ('T2', _DP), ('T3', _DP), ('T1', _DP),
                ('Ehead', _DP), ('Eend', _DP), ('alpha', _DP), ('alphaT', _DP), ('beta', _DP),
                ('betaT', _DP), ('gamma', _DP), ('phE', _DP), ('psiY', _DP), ('use_nco', C.POINTER(C.c_uint8)), ('out_sos', _DP),
                ('fm_interp', _DP), ('sos_Lseg', C.c_int32), ('sos_CA', _DP), ('sos_AP', _DP),
                ('tc_enable', C.c_int32), ('tc_K', C.c_int32), ('tc_isz', C.c_int32),
                ('tc_ncol', C.c_int32), ('tc_nout', C.c_int32), ('tc_npad', C.c_int32),
                ('tc_S', C.c_int32), ('tc_S_yl', C.c_int32), ('tc_nrowc', C.c_int32), ('tc_a_signed', C.c_int32),
                ('tc_Bq', C.POINTER(C.c_int8)), ('tc_cst', _DP), ('tc_rowc', _DP),
                ('tc_xor', C.c_uint8 * 16),
                ('lookahead', C.c_int32), ('fs', C.c_int64), ('chunk_step', C.POINTER(C.c_int64)),
                ('PN', _DP), ('sos_AM', _DP), ('sos_CAM', _DP),
                ('ssb_omega', C.c_double), ('ssb_rot', _DP)]


EXPORTS = ['sdrb_create', 'sdrb_destroy', 'sdrb_last_error', 'sdrb_outputs_per_chunk',
           'sdrb_chunk_bytes', 'sdrb_process', 'sdrb_process_device', 'sdrb_submit', 'sdrb_wait',
           'sdrb_get_iq_state', 'sdrb_set_iq_state', 'sdrb_read_decimated', 'sdrb_launch_count',
           'sdrb_fm_demod', 'sdrb_am_demod', 'sdrb_real_output', 'sdrb_imag_output',
           'sdrb_shift_freq', 'sdrb_power_spectrum', 'sdrb_stft_db', 'sdrb_global_error', 'sdrb_process_device_phases',
           'sdrb_set_profiling', 'sdrb_kernel_times', 'sdrb_keep_decimated', 'sdrb_read_debug', 'sdrb_iq_export_device',
           'sdrb_iq_prefix_device', 'sdrb_decode_iq', 'sdrb_correct_iq', 'sdrb_keep_x0', 'sdrb_read_x0', 'sdrb_iq_gain', 'sdrb_set_smooth', 'sdrb_host_alloc', 'sdrb_host_free', 'sdrb_reserve_sms',
           'sdrb_stream', 'sdrb_stream_device', 'sdrb_stream_end', 'sdrb_stream_end_device', 'sdrb_stream_lookahead',
           'sdrb_row_doubles', 'sdrb_iq_output', 'sdrb_ssb_demod',
           'sdrb_stream_samples', 'sdrb_stream_samples_device', 'sdrb_stream_samples_end',
           'sdrb_stream_samples_end_device', 'sdrb_stream_capacity']


def nvcc_command(out: str = LIB_PATH) -> list[str]:
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    return [nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
            '-Xcompiler', '-fPIC', '-shared', '-o', out, SOURCES[0]]


def build(force: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    stale = force or not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in SOURCES + [HEADER])
    if stale:
        env = dict(os.environ)
        env.pop('CC', None), env.pop('CXX', None)
        subprocess.run(nvcc_command(), check=True, env=env)
    return LIB_PATH


_lib = None


def lib():
    """The loaded library; raises SdrbError (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SdrbError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; '
                            f'g.build()"` (there is no CPU fallback)')
        L = C.CDLL(LIB_PATH)
        vp, sz = C.c_void_p, C.c_size_t
        L.sdrb_create.argtypes = [C.POINTER(Config), C.POINTER(Tables), C.POINTER(vp)]
        L.sdrb_destroy.argtypes = [vp]
        L.sdrb_last_error.argtypes = [vp]
        L.sdrb_last_error.restype = C.c_char_p
        L.sdrb_global_error.restype = C.c_char_p
        L.sdrb_outputs_per_chunk.argtypes = [vp]
        L.sdrb_row_doubles.argtypes = [vp]
        L.sdrb_chunk_bytes.argtypes = [vp]
        L.sdrb_chunk_bytes.restype = sz
        L.sdrb_process.argtypes = [vp, vp, sz, vp]
        L.sdrb_process_device.argtypes = [vp, vp, sz, vp, vp]
        L.sdrb_process_device_phases.argtypes = [vp, vp, sz, vp, vp, C.c_int]
        L.sdrb_set_profiling.argtypes = [vp, C.c_int]
        L.sdrb_kernel_times.argtypes = [vp, C.POINTER(C.c_float)]
        L.sdrb_submit.argtypes = [vp, C.c_int, vp, sz, vp]
        L.sdrb_wait.argtypes = [vp, C.c_int]
        L.sdrb_get_iq_state.argtypes = [vp, _DP]
        L.sdrb_set_iq_state.argtypes = [vp, _DP]
        L.sdrb_read_decimated.argtypes = [vp, sz, vp]
        L.sdrb_keep_decimated.argtypes = [vp, C.c_int]
        L.sdrb_read_debug.argtypes = [vp, vp]
        L.sdrb_iq_export_device.argtypes = [vp, vp, C.c_double, vp]
        L.sdrb_iq_prefix_device.argtypes = [vp, vp, C.c_int, vp]
        L.sdrb_launch_count.argtypes = [vp]
        L.sdrb_launch_count.restype = C.c_longlong
        for name in ('sdrb_fm_demod', 'sdrb_am_demod', 'sdrb_real_output', 'sdrb_imag_output', 'sdrb_iq_output'):
            getattr(L, name).argtypes = [C.c_int, vp, C.c_int, C.c_int, vp]
        L.sdrb_ssb_demod.argtypes = [C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, C.c_double, vp]
        L.sdrb_shift_freq.argtypes = [C.c_int, vp, vp, C.c_int, C.c_int, vp]
        L.sdrb_power_spectrum.argtypes = [C.c_int, vp, vp, C.c_int, C.c_int, vp]
        L.sdrb_stft_db.argtypes = [C.c_int, vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
        L.sdrb_decode_iq.argtypes = [C.c_int, vp, sz, C.c_char, C.c_int, vp]
        L.sdrb_correct_iq.argtypes = [C.c_int, vp, sz, _DP, C.c_double]
        L.sdrb_keep_x0.argtypes = [vp, C.c_int]
        L.sdrb_iq_gain.argtypes = [vp, vp, sz]
        L.sdrb_host_alloc.argtypes = [sz, C.POINTER(vp)]
        L.sdrb_host_free.argtypes = [vp]
        L.sdrb_reserve_sms.argtypes = [vp, C.c_int]
        L.sdrb_set_smooth.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
        L.sdrb_read_x0.argtypes = [vp, sz, vp]
        szp = C.POINTER(sz)
        L.sdrb_stream.argtypes = [vp, vp, sz, vp, szp]
        L.sdrb_stream_device.argtypes = [vp, vp, sz, vp, vp, szp]
        L.sdrb_stream_end.argtypes = [vp, vp, szp]
        L.sdrb_stream_end_device.argtypes = [vp, vp, vp, szp]
        L.sdrb_stream_lookahead.argtypes = [vp]
        L.sdrb_stream_samples.argtypes = [vp, vp, sz, vp, szp]
        L.sdrb_stream_samples_device.argtypes = [vp, vp, sz, vp, vp, szp]
        L.sdrb_stream_samples_end.argtypes = [vp, vp, szp]
        L.sdrb_stream_samples_end_device.argtypes = [vp, vp, vp, szp]
        L.sdrb_stream_capacity.argtypes = [vp, sz]
        L.sdrb_stream_capacity.restype = sz
        _lib = L
    return _lib


class PinnedBuffer:
    """Page-locked host memory from the library (cudaHostAlloc) with a numpy view."""

    def __init__(self, nbytes: int):
        import numpy as np
        self.ptr = C.c_void_p()
        check(lib().sdrb_host_alloc(nbytes, C.byref(self.ptr)))
        self.nbytes = nbytes
        self.u8 = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr.value))

    def view(self, dtype):
        return self.u8.view(dtype)

    def free(self):
        if self.ptr:
            lib().sdrb_host_free(self.ptr)
            self.ptr = C.c_void_p()
            self.u8 = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def check(rc: int, handle=None) -> None:
    if rc != 0:
        L = lib()
        msg = L.sdrb_last_error(handle) if handle else L.sdrb_global_error()
        raise SdrbError(f'libsdrterm_b200 error {rc}: {(msg or b"").decode(errors="replace")}')
