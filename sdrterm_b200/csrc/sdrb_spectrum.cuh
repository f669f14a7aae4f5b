// sdrb_spectrum.cuh -- the FFT feed of the reference's plot consumers, on the device.
//
//   k_gfft4 / k_gfft2   Stockham radix-4 / radix-2 passes of a batch of N-point complex FP64
//                       transforms between two global buffers (N = a chunk: 2^13 .. 2^17 samples;
//                       one launch per pass, the working set lives in L2); the first pass also
//                       applies the NCO vector (demodulation.py:71-79), twiddles by sincospi
//   k_spectrum_db       log10(|fftshift(X / N)|^2)                (spectrum_analyzer_plot.py:75-82)
//   k_stft_db           10 log10 |ShortTimeFFT.stft(y)|: one warp per slice, window * segment,
//                       zero-padded mfft-point transform in shared memory, centred (waterfall_plot.py:28-105)
//
// Reference behaviour reproduced: src/plots/spectrum_analyzer_plot.py:75-97 (`shiftFreq`, then
// `abs(fftshift(fftn(y, norm='forward')))`, `log10(amp*amp)`), src/plots/waterfall_plot.py:44-51,
// 97-99 (`ShortTimeFFT.from_window(('kaiser', 5), fs, 256, 128, mfft=1024, fft_mode='centered',
// scale_to='magnitude', phase_shift=None)`, `10*log10(abs(stft(y)))`).  The Qt widgets around them
// are not part of this build.
#pragma once
#include "sdrb_fft.cuh"
#include "sdrb_finish.cuh"

// One radix-4 Stockham pass: butterfly j of transform `blockIdx.y`; twiddle exp(-2 pi i k / (4 Ns)).
__global__ void __launch_bounds__(256)
k_gfft4(const double2 *__restrict__ in, double2 *__restrict__ out, const double2 *__restrict__ shift, int N, int Ns)
{
    const int quarter = N >> 2;
    const double2 *src = in + (size_t)blockIdx.y * N;
    double2 *dst = out + (size_t)blockIdx.y * N;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < quarter; j += gridDim.x * blockDim.x) {
        const int k = j & (Ns - 1);
        double2 a = src[j], b = src[j + quarter], c = src[j + 2 * quarter], d = src[j + 3 * quarter];
        if (shift) {                                   // first pass only: y * shift, elementwise
            a = cmul(a, shift[j]); b = cmul(b, shift[j + quarter]);
            c = cmul(c, shift[j + 2 * quarter]); d = cmul(d, shift[j + 3 * quarter]);
        }
        double2 w1 = make_double2(1.0, 0.0), w2 = w1, w3 = w1;      // k = 0: no sincospi, no products
        if (k) {
            const double x = -(double)k / (double)(2 * Ns);          // angle / pi of w1, exact
            sincospi(x, &w1.y, &w1.x);
            sincospi(2.0 * x, &w2.y, &w2.x);
            sincospi(3.0 * x, &w3.y, &w3.x);
        }
        fft_bfly4(a, b, c, d, w1, w2, w3, false, k != 0);
        const int j0 = ((j - k) << 2) + k;
        dst[j0] = a;
        dst[j0 + Ns] = b;
        dst[j0 + 2 * Ns] = c;
        dst[j0 + 3 * Ns] = d;
    }
}

// One radix-2 Stockham pass (the last one when log2 N is odd); twiddle exp(-2 pi i k / (2 Ns)).
__global__ void __launch_bounds__(256)
k_gfft2(const double2 *__restrict__ in, double2 *__restrict__ out, const double2 *__restrict__ shift, int N, int Ns)
{
    const int half = N >> 1;
    const double2 *src = in + (size_t)blockIdx.y * N;
    double2 *dst = out + (size_t)blockIdx.y * N;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < half; j += gridDim.x * blockDim.x) {
        const int k = j & (Ns - 1);
        double2 a = src[j], b = src[j + half];
        if (shift) { a = cmul(a, shift[j]); b = cmul(b, shift[j + half]); }
        double2 w = make_double2(1.0, 0.0);                          // k = 0: no sincospi, no product
        if (k) sincospi(-(double)k / (double)Ns, &w.y, &w.x);
        fft_bfly2(a, b, w, k != 0);
        const int j0 = ((j - k) << 1) + k;
        dst[j0] = a;
        dst[j0 + Ns] = b;
    }
}

// amp = |X[k]| / N after fftshift; out = log10(amp * amp)  (the reference's two statements).
__global__ void __launch_bounds__(256)
k_spectrum_db(const double2 *__restrict__ X, double *__restrict__ out, int N)
{
    const double2 *src = X + (size_t)blockIdx.y * N;
    double *dst = out + (size_t)blockIdx.y * N;
    const double inv = 1.0 / (double)N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double2 v = src[(i + ((N + 1) >> 1)) % N];                // fftshift: out[i] = X[(i + ceil(N/2)) mod N]
        const double amp = hypot(v.x * inv, v.y * inv);
        dst[i] = log10(amp * amp);
    }
}

// Short-time transform, one warp per slice p: seg[m] = y[p hop - mid + m] win[m] (zero outside
// the signal), zero-padded to mfft points, forward FFT in shared memory (fft on the warp), centred
// (out row q = bin (q + mfft/2) mod mfft), out[q][p] = 10 log10 |S|.
__global__ void __launch_bounds__(128)
k_stft_db(const double2 *__restrict__ y, const double2 *__restrict__ shift, const double *__restrict__ win, double *__restrict__ out,
          int n, int nperseg, int hop, int mid, int mfft, int p_num)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, W = blockDim.x >> 5;
    double2 *tw = reinterpret_cast<double2 *>(smem_raw);                 // exp(-2 pi i k / mfft), k < mfft/2
    for (int k = threadIdx.x; k < (mfft >> 1); k += blockDim.x) {
        double2 w;
        sincospi(-2.0 * (double)k / (double)mfft, &w.y, &w.x);
        tw[k] = w;
    }
    double2 *fa = tw + (mfft >> 1) + (size_t)warp * 2 * mfft, *fb = fa + mfft;
    __syncthreads();
    for (int p = blockIdx.x * W + warp; p < p_num; p += gridDim.x * W) {
        const long start = (long)p * hop - mid;
        for (int m = lane; m < mfft; m += 32) {
            double2 v = make_double2(0.0, 0.0);
            const long k = start + m;
            if (m < nperseg && k >= 0 && k < n) {
                v = y[k];
                if (shift) v = cmul(v, shift[k]);
                v = cscale(win[m], v);
            }
            fa[m] = v;
        }
        __syncwarp();
        const double2 *X = fft(fa, fb, mfft, mfft, false, tw, WarpGroup{lane});
        for (int qo = lane; qo < mfft; qo += 32) {
            const double2 v = X[(qo + (mfft >> 1)) & (mfft - 1)];
            out[(size_t)qo * p_num + p] = 10.0 * log10(hypot(v.x, v.y));
        }
        __syncwarp();
    }
}
