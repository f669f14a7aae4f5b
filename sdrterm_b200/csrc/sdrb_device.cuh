// sdrb_device.cuh -- device-side plan, small complex helpers, sample decode.
// Part of libsdrterm_b200.so (sm_100a).  See DESIGN.md section 3 for the algorithm.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define SDRB_TB 32          // blocks per tile == warp width (lane <-> block)
#define SDRB_NP 8           // poles of the cheby1 order-8 decimation low-pass
#define SDRB_XSTRIDE 33     // exchange buffer row stride in doubles
#define SDRB_NEDGE 320      // edge samples a chunk-boundary kernel stages: head (edge+1) + end window (nend)

enum { ENC_b = 0, ENC_B, ENC_h, ENC_H, ENC_i, ENC_I, ENC_f, ENC_d, ENC_Z };

struct DevPlan {
    int enc, itemsize, swap, correct_iq, normalize, demod, be_out;
    int q, N, edge, L, Mf, rem, M, ntiles, cnt_last, Hq, KS, R, nend, ws, k_bnd, nsec_out;
    int RL;                // pairs per DMMA k-lane (== KS): lane k owns pairs [k*RL, (k+1)*RL)
    int sb;                // bytes per complex sample
    int run_len[8];        // samples per run, sample order (4 ascending + 4 descending)
    int sos_ns, sos_Lseg;  // output SOS evaluated in 32 segments of sos_Lseg samples
    int fft_ok;            // FM resample by FFT (M == 2h, h power of two)
    int fft_n;             // twiddle table length (== M when fft_ok)
    int demod_in_smem;     // FFT / row buffers fit shared memory
    double Liq, lam, lam_q, lam_N, lam_inv, g0, d, norm_xmin, norm_k;
    double lam_run[8];     // lam^run_len
    double sos_AP[320];    // [5][ns][ns] (A^Lseg)^(2^lv), ns = sos_ns (packed): the lane scan's segment maps
    double lamq_pow[5];    // lam_q^(1,2,4,8,16)
    double lam_pw[33];     // lam^k, k = 0..32 (k_finish's IQ scans)
    double mu_pw[33];      // lam^-k
    double lam_tile[2];
    double2 p[SDRB_NP], P[SDRB_NP], rho[SDRB_NP], rho_p[SDRB_NP], c[SDRB_NP], zhat[SDRB_NP];
    double2 xi[SDRB_NP * SDRB_NP];
    double2 bx[SDRB_NP];   // p_i^edge / kappa_i: boundary vector -> anticausal carry (k_finish)
    double out_sos[4 * 6];
    const double *Afrag;   // [KS][2][32]  DMMA A fragments: even-part (Ec) and odd-part (Oc)
    const double *lam_j;   // [q+1]
    const double2 *Ppow;   // [TB+1][8]
    const double2 *pk;     // [edge+1][8]  p_i^k (closed forms of the head / tail recurrences)
    const double2 *Pt;     // [ntiles][8]  P_i^(32 m): a carry moved m whole tiles
    const double2 *RW;     // [TB+1][8]  rho_i   * P_i^l
    const double2 *RT;     // [TB+1][8]  rho_p_i * P_i^l
    const double2 *bnd;    // [M][8]
    const double2 *T2;     // [R][q]
    const double2 *T3;     // [R][TB+1]
    const double2 *T1;     // [R][ntiles]
    const double2 *Ehead;  // [R][edge+1]
    const double2 *Eend;   // [R][nend]
    // IQ corrector decoupled from the modal sums (DESIGN.md 3.3): the front ends sum the UNcorrected
    // rotated samples; with s[n] = off[n] e^{jwn} the true states are w_i = beta_i W~_i - alpha_i s,
    // T_i = betaT_i T~_i - alphaT_i s and y = sum rb_i W~_i + sum rbT_i T~_i + g0 u~ - gamma s
    const double2 *alpha;  // [R][8]  1 / (lam e^{jw} - p_i)
    const double2 *alphaT; // [R][8]  1 / (1 - p_i lam e^{jw})
    const double2 *beta;   // [R][8]
    const double2 *betaT;  // [R][8]
    const double2 *binv;   // [R][8]  1 / beta_i
    const double2 *binvT;  // [R][8]  1 / betaT_i
    const double2 *rb;     // [R][8]  rho_i beta_i
    const double2 *rbT;    // [R][8]  rho_i / p_i betaT_i
    const double2 *gamma;  // [R]     0 when the IQ correction is off
    const double2 *phE;    // [R]     e^{j w q Mf}
    const double2 *psiY;   // [2][R][TB]  gamma (lam e^{jw})^(q l): tile-start offset -> output of block l
    const double2 *Prot;   // [R][16]  rotating-frame block multipliers (8 forward, 8 backward)
    const double2 *tw;     // [fft_n]  exp(-2 pi i k / fft_n)
    const double *fm_interp;  // [M][M/2] or null
    const double *sos_CA;     // [sos_Lseg][ns]  c A^i
    const unsigned char *use_nco;  // [R]
    int W;                 // doubles per chunk-row of the output: 2M for iq ((Re, Im) pairs), M otherwise
    // usb / lsb: the band-pass h[m] e^{j Omega m} runs in the Weaver frame, u[k] = y[k] e^{-j Omega k}
    // through the real prototype out_sos (Re and Im alike), s[k] = Re(e^{j Omega k} v[k])
    double ssb_omega;      // +pi B / fs_d (usb), -pi B / fs_d (lsb); 0 otherwise
    const double2 *ssb_rot;   // [M+1] e^{j Omega k}, k = 0..M
};

// What a finish kernel instance writes: a real row from a demodulator (fm / am / re / im, output
// low-pass), the complex decimator output itself (iq), or the single-sideband audio (usb / lsb).
enum { OUT_REAL = 0, OUT_IQ = 1, OUT_SSB = 2 };

// ---------------------------------------------------------------- complex helpers (double2)
__device__ __forceinline__ double2 cmul(double2 a, double2 b)
{
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ double2 cfma(double2 a, double2 b, double2 c)  // a*b + c
{
    return make_double2(fma(a.x, b.x, fma(-a.y, b.y, c.x)), fma(a.x, b.y, fma(a.y, b.x, c.y)));
}
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 cconj(double2 a) { return make_double2(a.x, -a.y); }
__device__ __forceinline__ double2 cscale(double s, double2 a) { return make_double2(s * a.x, s * a.y); }

__device__ __forceinline__ double2 shfl_c(double2 v, int src)
{
    return make_double2(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src));
}
__device__ __forceinline__ double2 shfl_up_c(double2 v, int d)
{
    return make_double2(__shfl_up_sync(0xffffffffu, v.x, d), __shfl_up_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ double2 shfl_xor_c(double2 v, int m)
{
    return make_double2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}

// ---------------------------------------------------------------- affine scans o -> m o + a
// Inclusive composition of the lanes' maps across the warp, in place: lane l ends with the map of
// lanes 0..l, the later lane's map applied last.  The complex overload (multiplier mul) keeps the
// operand order of cmul, which does not round symmetrically.
__device__ __forceinline__ void warp_affine_scan(double &m, double2 &a, int lane)
{
#pragma unroll
    for (int lv = 0; lv < 5; lv++) {
        const double pm = __shfl_up_sync(0xffffffffu, m, 1 << lv);
        const double2 pa = shfl_up_c(a, 1 << lv);
        if (lane >= (1 << lv)) { a.x = fma(m, pa.x, a.x); a.y = fma(m, pa.y, a.y); m *= pm; }
    }
}
__device__ __forceinline__ void warp_affine_scan(double2 &mul, double2 &a, int lane)
{
#pragma unroll
    for (int lv = 0; lv < 5; lv++) {
        const double2 pa = shfl_up_c(a, 1 << lv), pm = shfl_up_c(mul, 1 << lv);
        if (lane >= (1 << lv)) { a = cfma(mul, pa, a); mul = cmul(mul, pm); }
    }
}

// The same across a CTA of up to 1024 threads: each thread's map (m, a) -> its exclusive map
// (em, ea), identity on thread 0, and the block total (tm, ta).  The warps' totals hop through
// s_m / s_a[32]; the caller syncs the block before it reuses them.
__device__ __forceinline__ void block_affine_scan(double m, double2 a, double *s_m, double2 *s_a,
                                                  double &em, double2 &ea, double &tm, double2 &ta)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    warp_affine_scan(m, a, lane);
    if (lane == 31) { s_a[warp] = a; s_m[warp] = m; }
    __syncthreads();
    if (warp == 0) {
        double wm = 1.0;
        double2 wa = make_double2(0.0, 0.0);
        if (lane < nw) { wm = s_m[lane]; wa = s_a[lane]; }
        warp_affine_scan(wm, wa, lane);
        s_a[lane] = wa; s_m[lane] = wm;
    }
    __syncthreads();
    // (warps before) then (lanes before in this warp)
    em = __shfl_up_sync(0xffffffffu, m, 1);
    ea = shfl_up_c(a, 1);
    if (lane == 0) { em = 1.0; ea = make_double2(0.0, 0.0); }
    if (warp > 0) {
        const double wm = s_m[warp - 1];
        const double2 wa = s_a[warp - 1];
        ea.x = fma(em, wa.x, ea.x); ea.y = fma(em, wa.y, ea.y); em *= wm;
    }
    tm = s_m[nw - 1]; ta = s_a[nw - 1];
}

// ---------------------------------------------------------------- decode (read_file.py:100-101)
// One complex sample n of a chunk: raw bytes -> (re, im) doubles, bit-exact for every integer
// encoding; float32 widens exactly.  `swap` = stored order differs from the GPU's little-endian.
template <int ENC>
__device__ __forceinline__ double2 load_sample(const uint8_t *__restrict__ raw, long n, int swap)
{
    if (ENC == ENC_b) {
        uint16_t v = *reinterpret_cast<const uint16_t *>(raw + 2 * n);
        return make_double2((double)(int8_t)(v & 0xff), (double)(int8_t)(v >> 8));
    } else if (ENC == ENC_B) {
        uint16_t v = *reinterpret_cast<const uint16_t *>(raw + 2 * n);
        return make_double2((double)(v & 0xff), (double)(v >> 8));
    } else if (ENC == ENC_h || ENC == ENC_H) {
        uint32_t v = *reinterpret_cast<const uint32_t *>(raw + 4 * n);
        if (swap) v = __byte_perm(v, 0, 0x2301);
        if (ENC == ENC_h)
            return make_double2((double)(int16_t)(v & 0xffff), (double)(int16_t)(v >> 16));
        return make_double2((double)(v & 0xffff), (double)(v >> 16));
    } else if (ENC == ENC_i || ENC == ENC_I || ENC == ENC_f) {
        uint2 v = *reinterpret_cast<const uint2 *>(raw + 8 * n);
        if (swap) { v.x = __byte_perm(v.x, 0, 0x0123); v.y = __byte_perm(v.y, 0, 0x0123); }
        if (ENC == ENC_i) return make_double2((double)(int32_t)v.x, (double)(int32_t)v.y);
        if (ENC == ENC_I) return make_double2((double)v.x, (double)v.y);
        return make_double2((double)__uint_as_float(v.x), (double)__uint_as_float(v.y));
    } else {  // ENC_d, ENC_Z: two doubles per sample
        ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(raw + 16 * n);
        if (swap && ENC == ENC_d) {
            uint32_t lo = (uint32_t)v.x, hi = (uint32_t)(v.x >> 32);
            v.x = ((unsigned long long)__byte_perm(lo, 0, 0x0123) << 32) | __byte_perm(hi, 0, 0x0123);
            lo = (uint32_t)v.y; hi = (uint32_t)(v.y >> 32);
            v.y = ((unsigned long long)__byte_perm(lo, 0, 0x0123) << 32) | __byte_perm(hi, 0, 0x0123);
        }
        return make_double2(__longlong_as_double((long long)v.x), __longlong_as_double((long long)v.y));
    }
}

// read_file.py:88-96 with the reference's operation order: ((1.6*(z - xmin))*k) - 0.8 on the
// real part, (1.6*im)*k on the imaginary part.
__device__ __forceinline__ double2 normalize_sample(double2 z, double xmin, double k)
{
    double re = __dmul_rn(__dmul_rn(1.6, __dadd_rn(z.x, -xmin)), k);
    double im = __dmul_rn(__dmul_rn(1.6, z.y), k);
    return make_double2(__dadd_rn(re, -0.8), im);
}

template <int ENC>
__device__ __forceinline__ double2 decode_sample(const DevPlan &pl, const uint8_t *__restrict__ raw, long n)
{
    double2 z = load_sample<ENC>(raw, n, pl.swap);
    if (pl.normalize) z = normalize_sample(z, pl.norm_xmin, pl.norm_k);
    return z;
}

// FP64 tensor-core MMA m8n8k4: D(8x8) += A(8x4) * B(4x8); A: row=lane>>2, col=lane&3;
// B: row=lane&3, col=lane>>2; C/D: row=lane>>2, cols 2*(lane&3)+{0,1}.  SASS: DMMA.8x8x4.
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
