/*
 * sdrterm_b200.h -- C ABI of libsdrterm_b200.so: the B200 (sm_100a) implementation of
 * peads/sdrterm's streamed IQ demodulation chain.
 *
 * The reference has no C ABI; its boundary is Python (SURVEY.md section 8b).  Each entry point
 * below names the reference interface it stands in for (paths relative to the reference tree).
 * All pointers are caller-owned; every function returns 0 on success and a negative code on
 * failure with a message available from sdrb_last_error(); nothing throws across the boundary.
 * A handle is not thread-safe: one handle per processor object, called from one thread.
 */
#ifndef SDRTERM_B200_H
#define SDRTERM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDRB_ABI_VERSION 11
#define SDRB_TILE_BLOCKS 32
#define SDRB_NPOLES 8
#define SDRB_MAX_DECIMATION 256

enum sdrb_status {
    SDRB_OK = 0,
    SDRB_ERR_ARG = -1,      /* bad argument / unsupported configuration */
    SDRB_ERR_CUDA = -2,     /* CUDA runtime error, see sdrb_last_error  */
    SDRB_ERR_NOMEM = -3,
    SDRB_ERR_STATE = -4
};

/* SDRB_IQ is not a reference mode: the complex decimator output y itself, 2 doubles (Re, Im) per
 * output, no output low-pass (n_out_sections 0), no --smooth-output. */
/* SDRB_USB / SDRB_LSB are not reference modes either: single-sideband audio.  With B = omegaOut
 * (0 < B < fs_d / 2, fs_d = fs / q) and the prototype h = ellip(3, 1, 30, B/2) at fs_d (out_sos,
 * n_out_sections 2), each row is s[k] = Re(sum_m h[m] e^{j Omega m} y[k-m]), Omega = +pi B / fs_d
 * (usb, the band [0, B] Hz) or -pi B / fs_d (lsb, [-B, 0] Hz): M doubles per chunk and row, from
 * a zero filter state per chunk (or once per stream in seamless mode). */
enum sdrb_demod { SDRB_FM = 0, SDRB_AM = 1, SDRB_RE = 2, SDRB_IM = 3, SDRB_IQ = 4, SDRB_USB = 5, SDRB_LSB = 6 };

/* Geometry and switches of one processor.  Mirrors the keyword arguments that
 * src/misc/io_args.py:97-141 passes to DspProcessor/VfoProcessor and to readFile
 * (src/misc/read_file.py:31-44). */
typedef struct sdrb_config {
    int32_t abi_version;     /* SDRB_ABI_VERSION */
    int32_t device;          /* CUDA device ordinal */
    char enc;                /* 'b','B','h','H','i','I','f','d' (file_util.py:46-60) or 'Z' =
                                already-decoded complex128 chunks (the Queue payload of
                                read_file.py:112) */
    uint8_t swap;            /* stored byte order differs from the host's (read_file.py:48-49,
                                file_util.py:92-95,106-107) */
    uint8_t correct_iq;      /* --correct-iq (read_file.py:55-77) */
    uint8_t normalize;       /* --normalize-input (read_file.py:79-96) */
    uint8_t demod;           /* enum sdrb_demod (io_args.py:37-47) */
    uint8_t big_endian_out;  /* SIMO framing '!d' (vfo_processor.py:84) vs '@d' (dsp_processor.py:162) */
    uint8_t seamless;        /* not a reference option: filter and demodulate the whole stream instead of
                                each chunk (sdrb_stream*; DESIGN.md section 11).  Needs q | N. */
    uint8_t reserved[1];
    int32_t q;               /* -d decimation, 2..SDRB_MAX_DECIMATION */
    int32_t N;               /* complex samples per chunk = 131072 / (2*itemsize) */
    int32_t edge;            /* sosfiltfilt pad length (27) */
    int32_t R;               /* rows: 1, or K+1 in --simo (vfo_processor.py:42-47) */
    int32_t n_out_sections;  /* output low-pass SOS sections (0 for re/im/iq; usb/lsb: the prototype's) */
    int32_t max_chunks;      /* largest number of chunks one sdrb_process* call will carry */
    double iq_L;             /* impedance / fs (read_file.py:65) */
    double norm_xmin;        /* read_file.py:177-196 */
    double norm_k;
} sdrb_config;

/* Host-computed tables (sdrterm_b200/plan.py; filter design is SciPy's as in
 * dsp_processor.py:39-45 and scipy.signal.decimate, the modal block form is derived from those
 * coefficients in extended precision).  Complex arrays are interleaved (re, im) doubles. */
typedef struct sdrb_tables {
    /* filter modes, SDRB_NPOLES each */
    const double *p, *P, *rho, *rho_p, *c, *zhat;
    const double *xi;        /* [8][8] complex */
    double g0, d;
    const double *Ec, *Oc;   /* [4][Hq] complex, Hq = ceil(q/2) */
    const double *Ppow;      /* [TILE_BLOCKS+1][8] complex */
    const double *pk;        /* [max(edge+1, edge+rem)][8] complex: p_i^k, rem = N mod q */
    const double *Pt;        /* [ntiles][8] complex: p_i^(q*TILE_BLOCKS*m) */
    const double *bx;        /* [8] complex: p_i^edge / kappa_i */
    const double *bnd;       /* [M][8] complex */
    int32_t k_bnd;
    /* IQ corrector */
    double lam, lam_q, lam_N, lam_inv;
    const double *lam_j;     /* [q+1] */
    const double *lam_k;     /* [33] lam^k */
    const double *mu_k;      /* [33] lam^-k */
    double lam_tile[2];
    int32_t RL;              /* pairs per DMMA k-lane = ceil(Hq/4) */
    int32_t run_len[8];      /* samples per run of a block, sample order */
    double lam_run[8];       /* lam^run_len */
    /* per row */
    const double *T2;        /* [R][q] complex */
    const double *T3;        /* [R][TILE_BLOCKS+1] complex */
    const double *T1;        /* [R][ntiles] complex */
    const double *Ehead;     /* [R][edge+1] complex */
    const double *Eend;      /* [R][nend] complex */
    /* IQ corrector decoupled from the block sums (DESIGN.md 3.3): per row and mode */
    const double *alpha, *alphaT; /* [R][8] complex */
    const double *beta, *betaT;   /* [R][8] complex */
    const double *gamma;          /* [R] complex (0 when --correct-iq is off) */
    const double *phE;            /* [R] complex: NCO phase at sample q*floor(N/q) */
    const double *psiY;           /* [2][R][TILE_BLOCKS] complex */
    const uint8_t *use_nco;      /* [R] 0 = no shift for this row (centre == 0, dsp_processor.py:185-187) */
    /* demodulation */
    const double *out_sos;   /* [n_out_sections][6] */
    const double *fm_interp; /* optional dense [M][M/2] matrix for non-power-of-two FM resample */
    int32_t sos_Lseg;        /* output SOS evaluated in 32 segments of this many samples */
    const double *sos_CA;    /* [sos_Lseg][ns], ns = 2*n_out_sections: c A^i */
    const double *sos_AP;    /* [5][ns][ns]: (A^Lseg)^(2^lv), lv = 0..4; required with an output SOS */
    /* tensor-core block front end (plan.py: build_tc); tc_enable == 0 selects the FP64 block
     * kernel.  The raw stream is the int8 A operand of an exact GEMM whose rows are super-blocks
     * of two blocks, against one tc_Bq slice per row of the bank. */
    int32_t tc_enable;
    int32_t tc_K;            /* bytes per GEMM row = 2 * q * 2 * itemsize (256 or 512) */
    int32_t tc_isz;          /* bytes per I or Q item */
    int32_t tc_ncol;         /* digit columns per fixed-point output (5) */
    int32_t tc_nout;         /* fixed-point outputs per row (40) */
    int32_t tc_npad;         /* GEMM N per row (208) */
    int32_t tc_S;            /* outputs 0..35 are integers * 2^-tc_S */
    int32_t tc_S_yl;         /* outputs 36..39 are integers * 2^-tc_S_yl */
    int32_t tc_nrowc;        /* complex constants per row in tc_rowc */
    int32_t tc_a_signed;     /* the GEMM reads the fixed-up raw bytes as signed (b, h) or unsigned (B, H) int8 */
    const int8_t *tc_Bq;     /* [R][tc_npad][tc_K] coefficient digits */
    const double *tc_cst;    /* [R][tc_nout + 4] */
    const double *tc_rowc;   /* [R][tc_nrowc] complex: epilogue constants (plan.py RC_* layout) */
    uint8_t tc_xor[16];      /* XOR pattern of 16 consecutive stream bytes */
    /* seamless streaming (cfg.seamless; plan.py build_plan(seamless=True)) */
    int32_t lookahead;       /* D: a chunk's output is final once the D chunks after it exist */
    int64_t fs;              /* sample rate in Hz (exact integer NCO phase across chunks) */
    const int64_t *chunk_step;   /* [R] (f_r * N) mod fs: NCO phase step per chunk, in units of 2 pi / fs */
    const double *PN;        /* [lookahead+1][8] complex: p_i^(N j) */
    const double *sos_AM;    /* [ns][ns]: A^M of the output cascade */
    const double *sos_CAM;   /* [M][ns]: c A^i, i < M */
    /* single sideband (SDRB_USB / SDRB_LSB).  The band-pass is the rotated prototype
     * (e^{j Omega} A, e^{j Omega} b, c, d); its segment and chunk maps are the real tables above times
     * powers of e^{j Omega}: A'^L = e^{j Omega L} A^L, c'A'^k = e^{j Omega k} c A^k.  The kernels hold
     * the 4 complex states in the frame of the chunk's first output (Weaver: y e^{-j Omega k} through
     * the real cascade), so they need only the rotations. */
    double ssb_omega;        /* Omega = +-pi B / fs_d */
    const double *ssb_rot;   /* [M+1] complex: e^{j Omega k}, k = 0..M (k = M: the seamless chunk map) */
} sdrb_tables;

typedef struct sdrb_handle sdrb_handle;

/* Stands in for constructing a DspProcessor/VfoProcessor and selecting its demodulation
 * (src/dsp/dsp_processor.py:51-138, src/dsp/vfo_processor.py:38-69). */
int sdrb_create(const sdrb_config *cfg, const sdrb_tables *tab, sdrb_handle **out);
int sdrb_destroy(sdrb_handle *h);
const char *sdrb_last_error(const sdrb_handle *h);

/* Geometry derived from the config: outputs per chunk-row M = ceil(N/q), bytes per chunk, and the
 * doubles per chunk-row of the output buffers W (2M for SDRB_IQ: (Re, Im) interleaved, M otherwise). */
int sdrb_outputs_per_chunk(const sdrb_handle *h);
size_t sdrb_chunk_bytes(const sdrb_handle *h);
int sdrb_row_doubles(const sdrb_handle *h);

/* The hot path: feedBuffers' decode/normalise/IQ-correct (src/misc/read_file.py:100-103) +
 * DspProcessor._processChunk (src/dsp/dsp_processor.py:140-149) + framing (:162,
 * vfo_processor.py:84) over `nchunks` whole chunks.
 *   raw : nchunks * chunk_bytes bytes
 *   out : R * nchunks * W doubles, row-major [row][chunk][W] (each row is one output stream; W =
 *         sdrb_row_doubles); byte-swapped to big-endian when cfg.big_endian_out
 * sdrb_process takes HOST buffers (pinned or pageable) and includes H2D/D2H; it returns after
 * the results are in `out`.  sdrb_process_device takes DEVICE buffers and only enqueues work on
 * `stream` (a cudaStream_t, may be NULL). */
int sdrb_process(sdrb_handle *h, const void *raw, size_t nchunks, double *out);
int sdrb_process_device(sdrb_handle *h, const void *raw_dev, size_t nchunks, double *out_dev,
                        void *stream);

/* The same chain split for time-segment sharding across GPUs (SURVEY.md section 8e): phase bits
 * 1 = block kernel, 2 = IQ-offset scan from the handle's IQ state, 4 = fix-up + demodulation.
 * A rank runs (1|2|8) from a zero state, exports its segment's offset gain, the ranks exchange
 * gains, each folds the ones before it into its initial state and runs (2|4); the raw data is
 * read once. */
#define SDRB_PHASE_MAIN 1
#define SDRB_PHASE_IQSCAN 2
#define SDRB_PHASE_FINISH 4
#define SDRB_PHASE_ZERO_IQ 8   /* clear the IQ state (on the stream) before anything else */
int sdrb_process_device_phases(sdrb_handle *h, const void *raw_dev, size_t nchunks, double *out_dev,
                               void *stream, int phases);

/* The exchange between the two passes without a host round trip: export this segment's gained
 * offset and length as 3 doubles (re, im, nsamples) into a device buffer the caller all-gathers,
 * then fold the gains of ranks 0..rank-1 ([world][3] doubles) into this handle's IQ state. */
int sdrb_iq_export_device(sdrb_handle *h, double *dst3_dev, double nsamples, void *stream);
int sdrb_iq_prefix_device(sdrb_handle *h, const double *gains3_dev, int rank, void *stream);

/* --smooth-output (src/dsp/dsp_processor.py:159-160): after the output low-pass, every chunk's row of
 * M outputs goes through scipy.signal.savgol_filter(z, window, 3) as three linear maps taken from
 * SciPy itself: outputs 0..nhead-1 = head rows applied to the first `window` samples, outputs
 * M-ntail..M-1 = tail rows applied to the last `window` samples, every other output k = the FIR row
 * applied to samples k+lo .. k+lo+window-1.  `tab` is [nhead + 1 + ntail][window] doubles (head rows,
 * FIR row, tail rows); window 0 switches smoothing off.  Native-endian output only (the SIMO path of
 * the reference never smooths).  SDRB_IQ output is never smoothed: SDRB_ERR_ARG. */
int sdrb_set_smooth(sdrb_handle *h, int window, int nhead, int ntail, int lo, const double *tab);

/* Pre-pass of time-segment sharding for segments longer than one batch: advance the IQ state over
 * `nchunks` raw HOST chunks exactly as sdrb_process would, without computing any output (the
 * offset a segment gains from a zero state is what the ranks exchange, SURVEY 8e). */
int sdrb_iq_gain(sdrb_handle *h, const void *raw_host, size_t nchunks);

/* CUDA-event timing of the kernel groups of the last full sdrb_process_device call: ms[0] = block
 * front end (k_tc / k_main), ms[1] = IQ-offset kernels, ms[2] = k_finish (or k_fixup), ms[3] =
 * k_demod (general path only, 0 otherwise); for bench.py's roofline. */
int sdrb_set_profiling(sdrb_handle *h, int on);
int sdrb_kernel_times(sdrb_handle *h, float ms[4]);

/* Double-buffered streaming from pinned host memory: sdrb_submit enqueues H2D + kernels + D2H for
 * one batch on slot (0 or 1) and returns; sdrb_wait blocks until that slot's `out` (R * nchunks * W
 * doubles, laid out as for sdrb_process) is complete.
 * Batches must be submitted in stream order; the IQ-corrector state chains through them. */
int sdrb_submit(sdrb_handle *h, int slot, const void *raw_host, size_t nchunks, double *out_host);
int sdrb_wait(sdrb_handle *h, int slot);

/* The persistent kernels (k_tc, k_finish) normally take every SM.  When a collective runs beside
 * them (the NCCL broadcast of the next raw batch in a row-sharded bank), leave `nsm` SMs free so
 * that its thread blocks can be scheduled and the transfer really overlaps the kernels. */
int sdrb_reserve_sms(sdrb_handle *h, int nsm);

/* Page-locked host staging buffers for sdrb_submit (so that a host layer needs nothing but this
 * library to stream: the drop-in CLI does not import torch). */
int sdrb_host_alloc(size_t bytes, void **ptr_out);
int sdrb_host_free(void *ptr);

/* The one piece of state that crosses chunks: the IQ corrector's complex offset
 * (src/misc/read_file.py:53).  Used for time-segment sharding across GPUs. */
int sdrb_get_iq_state(sdrb_handle *h, double off[2]);
int sdrb_set_iq_state(sdrb_handle *h, const double off[2]);

/* Test/diagnostic access: complex decimator output of the last batch, [chunk][row][M]
 * interleaved doubles (what `y` holds after dsp_processor.py:147). */
int sdrb_read_decimated(sdrb_handle *h, size_t nchunks, double *y_host);
/* The fused finish kernel keeps y on chip; it is written out only when this is switched on
 * (off by default; the general k_fixup/k_demod path always writes it). */
int sdrb_keep_decimated(sdrb_handle *h, int on);
/* Diagnostic: clock64 timelines of CTA 0 -- k_tc's pipeline [32 tiles][16 events] in the first 512
 * values, k_finish's phases [16 items][16 events] in the second 512 (microbench/tc_timeline.py);
 * needs the environment variable SDRB_TC_DEBUG=1 when the handle is created. */
int sdrb_read_debug(sdrb_handle *h, unsigned long long *out1024);

/* Kernel launches issued by this handle since creation (bench.py's gpu_launches). */
long long sdrb_launch_count(const sdrb_handle *h);

/* Module-level operators of src/dsp/demodulation.py (caller-owned in/out host arrays):
 *   sdrb_fm_demod   fmDemod(data(R,M) c128, out(R,M) f64)        demodulation.py:25-38
 *   sdrb_am_demod   amDemod                                       demodulation.py:41-48
 *   sdrb_real_output / sdrb_imag_output                           demodulation.py:51-68
 *   sdrb_iq_output  y(R,M) c128 -> out(R,2M) f64, (Re, Im) interleaved (not a reference operator)
 *   sdrb_ssb_demod  y(R,M) c128 -> out(R,M) f64: s = Re(e^{j omega k} sosfilt(sos, y e^{-j omega k})),
 *                   the single-sideband band-pass of the prototype sos ([nsec][6], nsec 1..4) rotated
 *                   by omega (0 < |omega| < pi/2), zero state per row, any M (not a reference operator)
 *   sdrb_shift_freq shiftFreq(y(N), shift(R,N), res(R,N))         demodulation.py:71-79 */
int sdrb_fm_demod(int device, const double *y, int R, int M, double *out);
int sdrb_am_demod(int device, const double *y, int R, int M, double *out);
int sdrb_real_output(int device, const double *y, int R, int M, double *out);
int sdrb_imag_output(int device, const double *y, int R, int M, double *out);
int sdrb_iq_output(int device, const double *y, int R, int M, double *out);
int sdrb_ssb_demod(int device, const double *y, int R, int M, const double *sos, int nsec, double omega, double *out);
int sdrb_shift_freq(int device, const double *y, const double *shift, int R, int N, double *res);
/* sdrb_fm_demod takes any even row length: 2*2^k rows run the FFT interpolation, other lengths a
 * dense scipy.signal.resample matrix built on the host in extended precision. */

/* The FFT feed of the reference's plot consumers (SURVEY 8-f3), caller-owned host arrays:
 *   sdrb_power_spectrum  SpectrumAnalyzerPlot.update, src/plots/spectrum_analyzer_plot.py:75-82:
 *       shiftFreq(y, shift, y); amp = abs(fftshift(fftn(y, norm='forward'))); amp = log10(amp*amp)
 *       y: `batch` rows of N complex128 (N a power of two >= 4: every chunk of the standard
 *       encodings is), shift: N complex128 applied to every row, or NULL; out: batch*N doubles.
 *   sdrb_stft_db         WaterfallPlot.update, src/plots/waterfall_plot.py:44-51,97-99:
 *       10*log10(abs(ShortTimeFFT.stft(y))) for fft_mode='centered', phase_shift=None; `win` is the
 *       ShortTimeFFT's (already scaled) window of nperseg values, slices p = 0..p_num-1 start at
 *       p*hop - nperseg/2, zero outside the n samples, zero-padded to mfft (power of two <= 4096);
 *       out: mfft rows of p_num doubles.  shift: n complex128 or NULL. */
int sdrb_power_spectrum(int device, const double *y, const double *shift, int N, int batch, double *out);
int sdrb_stft_db(int device, const double *y, const double *shift, int n, const double *win, int nperseg, int hop,
                 int mfft, int p_num, double *out);

/* The decode step of feedBuffers on its own (src/misc/read_file.py:100-101): the structured view
 * [('re',T),('im',T)] of `raw` -> interleaved complex128, bit-exact for every encoding; `swap` =
 * stored byte order differs from little-endian.  nsamples complex samples in, 2*nsamples doubles out. */
int sdrb_decode_iq(int device, const void *raw, size_t nsamples, char enc, int swap, double *z_out);

/* The reference's compiled-plugin seam, dsp.fast.iq_correction.IQCorrection.correctIq(data, off)
 * (extra/src/iq_correction.pyx:37-70, picked up by src/misc/read_file.py:58-63): in place on
 * nsamples interleaved complex128 values, `off_inout` is the corrector's carried complex offset,
 * L = impedance / fs. */
int sdrb_correct_iq(int device, double *z_inout, size_t nsamples, double off_inout[2], double L);

/* Test access to the tensor-core front end's integer decode: when switched on, the kernel also
 * stores the first raw sample of every block (two unit-coefficient outputs of the int8 GEMM,
 * exact integers) as [chunk][row][N/q] interleaved complex128. */
int sdrb_keep_x0(sdrb_handle *h, int on);
int sdrb_read_x0(sdrb_handle *h, size_t nchunks, double *x0_host);
/* Seamless streaming (not a reference option; DESIGN.md section 11).  On a handle created with
 * cfg.seamless the chunk stream is filtered and demodulated as ONE signal, the way
 * scipy.signal.decimate / sosfilt would treat the concatenated stream: the NCO phase runs on across
 * chunks, the decimator's zero-phase filter sees the stream's two real ends only, the fm
 * discriminator and the output low-pass carry their state.  The framing per chunk is unchanged
 * (W doubles per chunk and row, [row][chunk][W], big-endian when cfg.big_endian_out).
 *   sdrb_stream         host `raw` of nchunks whole chunks in; emits every chunk that has become final
 *                       (a chunk is final once the lookahead D chunks after it exist), synchronously,
 *                       into host `out` (room for nchunks + D chunks of R * W doubles each);
 *                       *nchunks_out = chunks emitted
 *   sdrb_stream_device  the same on device buffers, only enqueued on `stream` (`out_dev`: room for
 *                       nchunks chunks)
 *   sdrb_stream_end     end of stream: emits the chunks still held back, with the stream's real end
 *                       as the boundary (room for D chunks), and resets the stream (IQ offset included)
 *   sdrb_stream_end_device  the same into a device buffer, enqueued on `stream`
 *   sdrb_stream_lookahead   D
 * sdrb_process*, sdrb_submit, the phase entry points and sdrb_iq_gain return SDRB_ERR_STATE on such a
 * handle; sdrb_set_smooth returns SDRB_ERR_ARG (Savitzky-Golay per chunk is chunk-local by design). */
int sdrb_stream(sdrb_handle *h, const void *raw_host, size_t nchunks, double *out_host, size_t *nchunks_out);
int sdrb_stream_device(sdrb_handle *h, const void *raw_dev, size_t nchunks, double *out_dev, void *stream,
                       size_t *nchunks_out);
int sdrb_stream_end(sdrb_handle *h, double *out_host, size_t *nchunks_out);
int sdrb_stream_end_device(sdrb_handle *h, double *out_dev, void *stream, size_t *nchunks_out);
int sdrb_stream_lookahead(const sdrb_handle *h);
/* Sample-granular seamless streaming: any whole number of complex samples per call, for every q.
 * The handle's "chunk" (cfg.N) is then the seamless FRAME, a whole number of tiles (plan.py
 * seamless_frame_samples: 32 q floor(N_reader / (32 q)); the reader's chunk itself for a power-of-two
 * q).  The handle keeps the samples that do not fill a frame (fewer than N) on the device, in front
 * of the next call's samples; whole frames go through the sdrb_stream machinery.  Outputs are
 * counted per row: *nout outputs per row, `out` is [row][*nout * W / M] doubles, contiguous per row
 * (for whole frames exactly the [row][chunk][W] layout of sdrb_stream).
 *   sdrb_stream_samples         host `raw` of nsamples samples (at most max_chunks * N), synchronous
 *   sdrb_stream_samples_device  the same from a device buffer (one device-to-device copy into the
 *                               handle's window), only enqueued on `stream`
 *   sdrb_stream_samples_end     end of stream: the frames still held back and the partial last frame
 *                               (ceil(Lp / q) outputs from its Lp samples; scipy.signal.decimate's last
 *                               output of a ragged stream), then a reset.  A stream of 27 samples or
 *                               fewer (the decimator's pad length) is refused with SDRB_ERR_ARG.
 *   sdrb_stream_samples_end_device  the same into a device buffer
 *   sdrb_stream_capacity        the most outputs per row that a sdrb_stream_samples* call with
 *                               `nsamples` new samples, or an end call, can emit (size `out` by it)
 * A stream takes its input either in chunks (sdrb_stream*) or in samples (sdrb_stream_samples*): an
 * input call of the other kind returns SDRB_ERR_STATE until the stream ends, and so does
 * sdrb_stream_end while samples of a partial frame are pending.  An fm stream of at most q samples
 * (one output, no discriminator pair) is refused with SDRB_ERR_ARG at its end.
 * The first sample call allocates the handle's two raw windows ((max_chunks + 1) * N samples each).
 * An end call with a partial frame derives that frame's tables on the host and copies them from
 * pageable memory, which synchronises `stream` before the copy; the other sample calls only
 * enqueue. */
int sdrb_stream_samples(sdrb_handle *h, const void *raw_host, size_t nsamples, double *out_host, size_t *nout);
int sdrb_stream_samples_device(sdrb_handle *h, const void *raw_dev, size_t nsamples, double *out_dev, void *stream,
                               size_t *nout);
int sdrb_stream_samples_end(sdrb_handle *h, double *out_host, size_t *nout);
int sdrb_stream_samples_end_device(sdrb_handle *h, double *out_dev, void *stream, size_t *nout);
size_t sdrb_stream_capacity(const sdrb_handle *h, size_t nsamples);

const char *sdrb_global_error(void);

#ifdef __cplusplus
}
#endif
#endif /* SDRTERM_B200_H */
