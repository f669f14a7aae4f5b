// sdrb_fft.cuh -- the FFT every kernel shares (k_finish, k_demod, k_stft_db; k_gfft4 / k_gfft2 take
// the butterflies), and the FM 2x interpolation built on it.  Twiddles come from the half table
// tw[m] = exp(-2 pi i m / M), m < M/2, of the row length M.
#pragma once
#include "sdrb_device.cuh"

// The thread groups a transform runs on: rank, size and a barrier.
struct WarpGroup {
    int rank;
    static constexpr int size = 32;
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};
struct CtaGroup {
    int rank, size;
    __device__ __forceinline__ void sync() const { __syncthreads(); }
};

// exp(-+2 pi i m / M) for m < M from the half table tw[m], m < M/2 (tw[m + M/2] = -tw[m]).
__device__ __forceinline__ double2 fft_tw(const double2 *tw, int m, int Mh, bool inverse)
{
    const bool neg = m >= Mh;
    double2 w = tw[neg ? m - Mh : m];
    if (neg) { w.x = -w.x; w.y = -w.y; }
    if (inverse) w.y = -w.y;
    return w;
}

// Radix-4 butterfly with its twiddles w1..w3 (already conjugated for the inverse), in place: a..d
// become outputs 0..3.  twiddle = false: the twiddles are 1 and the products are skipped.
__device__ __forceinline__ void fft_bfly4(double2 &a, double2 &b, double2 &c, double2 &d, double2 w1, double2 w2,
                                          double2 w3, bool inverse, bool twiddle = true)
{
    if (twiddle) { b = cmul(w1, b); c = cmul(w2, c); d = cmul(w3, d); }
    const double2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = csub(b, d);
    // -i (b - d) forward, +i (b - d) inverse
    const double2 r3 = inverse ? make_double2(-s3.y, s3.x) : make_double2(s3.y, -s3.x);
    a = cadd(s0, s2);
    b = cadd(s1, r3);
    c = csub(s0, s2);
    d = csub(s1, r3);
}

// Radix-2 butterfly with twiddle w, in place (twiddle = false: w is 1, no product).
__device__ __forceinline__ void fft_bfly2(double2 &a, double2 &b, double2 w, bool twiddle = true)
{
    const double2 t = twiddle ? cmul(w, b) : b;
    b = csub(a, t);
    a = cadd(a, t);
}

// Stockham radix-4 pass over n points: one butterfly per thread and step; the twiddle
// exp(-+2 pi i k / (4 Ns)) = table entry k * tstride (table base M = 2 * Mh).
template <class G>
__device__ __forceinline__ void fft_pass4(const double2 *in, double2 *out, int n, int Ns, int tstride, bool inverse,
                                          const double2 *tw, int Mh, G g)
{
    const int quarter = n >> 2;
    for (int j = g.rank; j < quarter; j += g.size) {
        const int k = j & (Ns - 1);
        const int m = k * tstride;
        double2 a = in[j], b = in[j + quarter], c = in[j + 2 * quarter], d = in[j + 3 * quarter];
        fft_bfly4(a, b, c, d, fft_tw(tw, m, Mh, inverse), fft_tw(tw, 2 * m, Mh, inverse), fft_tw(tw, 3 * m, Mh, inverse),
                  inverse);
        const int j0 = ((j - k) << 2) + k;
        out[j0] = a;
        out[j0 + Ns] = b;
        out[j0 + 2 * Ns] = c;
        out[j0 + 3 * Ns] = d;
    }
}

// Stockham radix-2 pass over n points (two butterflies in flight per thread); twiddle
// exp(-+2 pi i k / (2 Ns)) = tw[k * tstride].
template <class G>
__device__ __forceinline__ void fft_pass2(const double2 *in, double2 *out, int n, int Ns, int tstride, bool inverse,
                                          const double2 *tw, G g)
{
    const int half = n >> 1;
    for (int j = g.rank; j < half; j += 2 * g.size) {
        const int jb = j + g.size;
        const bool two = jb < half;
        const int ka = j & (Ns - 1), kb = jb & (Ns - 1);
        double2 wa = tw[ka * tstride], wb = tw[kb * tstride];
        if (inverse) { wa.y = -wa.y; wb.y = -wb.y; }
        double2 a0 = in[j], a1 = in[j + half];
        double2 b0 = two ? in[jb] : a0, b1 = two ? in[jb + half] : a1;
        fft_bfly2(a0, a1, wa);
        fft_bfly2(b0, b1, wb);
        const int ja = ((j - ka) << 1) + ka, jc = ((jb - kb) << 1) + kb;
        out[ja] = a0;
        out[ja + Ns] = a1;
        if (two) {
            out[jc] = b0;
            out[jc + Ns] = b1;
        }
    }
}

// n-point FFT (n a power of two, n divides M) by radix-4 passes and one radix-2 pass if needed,
// with a barrier of the group after each; returns the buffer that holds the result.
template <class G>
__device__ __forceinline__ double2 *fft(double2 *src, double2 *dst, int n, int M, bool inverse, const double2 *tw, G g)
{
    int Ns = 1;
    for (; Ns * 4 <= n; Ns <<= 2) {
        fft_pass4(src, dst, n, Ns, M / (4 * Ns), inverse, tw, M >> 1, g);
        g.sync();
        double2 *tmp = src; src = dst; dst = tmp;
    }
    if (Ns < n) {
        fft_pass2(src, dst, n, Ns, M / (2 * Ns), inverse, tw, g);
        g.sync();
        double2 *tmp = src; src = dst; dst = tmp;
    }
    return src;
}

// scipy.signal.resample(ph, M) of the h = M/2 pair phases in fa (as doubles), h a power of two >= 2:
// the even outputs are the phases themselves (the caller stores them), the odd ones come from the
// half-sample-shifted spectrum.  Forward FFT of z[m] = ph[2m] + i ph[2m+1] at n2 = h/2 points, the
// shift, the inverse at n2 points; store_odd(k, v) takes output k = 4m+1, 4m+3.  fa and fb are n2
// points each and both are overwritten; the caller syncs before reading what store_odd wrote.
template <class G, class Store>
__device__ __forceinline__ void fm_interp2x(double2 *fa, double2 *fb, int M, const double2 *tw, G g, Store store_odd)
{
    const int h = M >> 1, n2 = M >> 2;
    double2 *src = fft(fa, fb, n2, M, false, tw, g);
    double2 *dst = src == fa ? fb : fa;
    // spectrum of the real row X[k] (k <= h/2) from Z, times the half-sample shift
    // H[k] = exp(i pi k / h), re-packed for the half-length inverse transform
    for (int k = g.rank; k <= (n2 >> 1); k += g.size) {
        if (k == 0) {
            const double2 Z0 = src[0];
            const double X0 = Z0.x + Z0.y;
            dst[0] = make_double2(X0, X0);
        } else {
            const int kp = n2 - k;
            const double2 Zk = src[k], Zc = cconj(src[kp]);
            const double2 Xe = cscale(0.5, cadd(Zk, Zc));
            const double2 dd = csub(Zk, Zc);
            const double2 Xo = make_double2(0.5 * dd.y, -0.5 * dd.x);           // -i (Zk - Zc) / 2
            const double2 w2 = tw[2 * k];                                       // exp(-2 pi i k / h)
            const double2 tX = cmul(w2, Xo);
            const double2 Xk = cadd(Xe, tX), Xkp = cconj(csub(Xe, tX));
            const double2 Uk = cmul(Xk, cconj(tw[k])), Ukp = cmul(Xkp, cconj(tw[kp]));
            // V[k] = (U[k] + conj U[k']) + i (U[k] - conj U[k']) conj(w2)
            const double2 s1 = cadd(Uk, cconj(Ukp)), d1 = cmul(csub(Uk, cconj(Ukp)), cconj(w2));
            dst[k] = make_double2(s1.x - d1.y, s1.y + d1.x);
            // V[k'] = (U[k'] + conj U[k]) + i (U[k'] - conj U[k]) (-w2)
            const double2 s2 = cadd(Ukp, cconj(Uk)), d2 = cmul(csub(Ukp, cconj(Uk)), w2);
            dst[kp] = make_double2(s2.x + d2.y, s2.y - d2.x);
        }
    }
    g.sync();
    src = fft(dst, src, n2, M, true, tw, g);
    const double sc1 = 1.0 / (double)h;
    for (int m = g.rank; m < n2; m += g.size) {
        const double2 v = src[m];
        store_odd(4 * m + 1, v.x * sc1);
        store_odd(4 * m + 3, v.y * sc1);
    }
}
