// sdrb_finish.cuh -- k_finish: everything after the block front end, one warp per (chunk, row).
//
//   1. chunk boundaries: IQ-corrected, NCO-shifted head and end-window samples; sosfiltfilt's odd
//      extension and zi start-up (head), the tail extension (end), the boundary vector zeta
//   2. carries of the 8 forward / 8 anticausal modal states across the tiles of the chunk
//   3. decimated outputs y[k] = partial output of the front end + carry-in response (+ boundary)
//   4. demodulation: fm (pair phase, 2x trigonometric interpolation by a real-input FFT of half
//      the length and its inverse) | am | re | im; the iq instance (OUT_IQ) stores y straight from
//      registers instead, (Re, Im) per output, and skips 3b-5
//   5. output low-pass (zero initial state per chunk): sdrb_outstage.cuh's output stage, 32 lane
//      segments composed by a Kogge-Stone scan of the segment maps; framing (native or big-endian)
//   The usb / lsb instance (OUT_SSB) skips 3b and 4: it stages y in the warp's shared memory (Re in
//   zrow, Im in the carry rows as they fall dead) and runs the same output stage on complex states
//   (the band-pass in the Weaver frame), then frames the real part.
//
// It replaces k_fixup + k_demod for the common shapes (whole tiles, M a power of two <= 1024, at
// most 2 output sections); those two kernels remain the general path.  Nothing leaves the SM
// between the stages: y, the phase row and the filtered row live in the warp's shared memory.
//
// Reference behaviour reproduced: scipy.signal.decimate's sosfiltfilt boundary handling
// (src/dsp/dsp_processor.py:147), src/dsp/demodulation.py:25-68, dsp_processor.py:32-36,149,162,
// src/dsp/vfo_processor.py:84, src/misc/read_file.py:65-77.  tests/emulator.py (emu_fixup,
// emu_demod, emu_fm_interp_real) is the numpy twin.
#pragma once
#include "sdrb_kernels.cuh"
#include "sdrb_outstage.cuh"

#define FIN_WARPS 8      // two CTAs of eight warps per SM: the per-CTA table set-up is paid twice per SM, not four times
#define FIN_DBG(ev) do { if (sc.dbg && blockIdx.x == 0 && warp == 0 && lane == 0 && nit < 16) sc.dbg[512 + nit * 16 + (ev)] = clock64(); } while (0)

// Per-warp shared memory (bytes); per CTA: twiddles exp(-2 pi i k / M) (k < M/2) and the pole
// powers p_i^k (k <= edge).
__host__ __device__ inline size_t finish_warp_bytes(int M)
{
    const int nt = M / SDRB_TB;
    size_t b = (size_t)(nt + 1) * 16 * sizeof(double2);      // carry; the second FFT buffer fb aliases it (carry is dead by then)
    size_t rest = (size_t)(M / 4) * sizeof(double2);         // fa
    rest += (size_t)(M + 32) * sizeof(double);               // zrow, one pad per segment
    // the phase-1 scratch overlays fa + zrow: addv [nt][16], then seqA[32], seqB[32] -- for rows of
    // 128 outputs and fewer it is the larger of the two
    const size_t scratch = ((size_t)nt * 16 + 64) * sizeof(double2);
    return b + (rest > scratch ? rest : scratch);
}
__host__ __device__ inline size_t finish_smem_bytes(int M, int edge)
{
    const int nt = M / SDRB_TB;
    const size_t tables = (size_t)(nt + 48 + nt * 8 + 32 + 32 + 64) * sizeof(double2);   // single-row tables
    return (size_t)(M / 2) * sizeof(double2) + (size_t)(edge + 1) * 8 * sizeof(double2) + tables + FIN_WARPS * finish_warp_bytes(M);
}

// Stockham radix-2 pass over n points by one warp (two butterflies in flight per lane); twiddle
// exp(-+2 pi i k / (2 Ns)) = tw[k * tstride].
__device__ __forceinline__ void fin_fft_pass(const double2 *in, double2 *out, int n, int Ns, int tstride,
                                             bool inverse, const double2 *tw, int lane)
{
    const int half = n >> 1;
    for (int j = lane; j < half; j += 64) {
        const int jb = j + 32;
        const bool two = jb < half;
        const int ka = j & (Ns - 1), kb = jb & (Ns - 1);
        double2 wa = tw[ka * tstride], wb = tw[kb * tstride];
        if (inverse) { wa.y = -wa.y; wb.y = -wb.y; }
        const double2 a0 = in[j], a1 = in[j + half];
        const double2 b0 = two ? in[jb] : a0, b1 = two ? in[jb + half] : a1;
        const double2 ta = cmul(wa, a1), tb = cmul(wb, b1);
        const int ja = ((j - ka) << 1) + ka, jc = ((jb - kb) << 1) + kb;
        out[ja] = cadd(a0, ta);
        out[ja + Ns] = csub(a0, ta);
        if (two) {
            out[jc] = cadd(b0, tb);
            out[jc + Ns] = csub(b0, tb);
        }
    }
}

// exp(-+2 pi i m / M) for m < M from the half table tw[m], m < M/2 (tw[m + M/2] = -tw[m]).
__device__ __forceinline__ double2 fin_tw(const double2 *tw, int m, int Mh, bool inverse)
{
    const bool neg = m >= Mh;
    double2 w = tw[neg ? m - Mh : m];
    if (neg) { w.x = -w.x; w.y = -w.y; }
    if (inverse) w.y = -w.y;
    return w;
}

// Stockham radix-4 pass over n points by one warp: one butterfly per lane and step; the twiddle
// exp(-+2 pi i k / (4 Ns)) = table entry k * tstride (table base M = 2 * Mh).  Half the passes of
// the radix-2 version, and each pass is one shared-memory round trip of dependent latency.
__device__ __forceinline__ void fin_fft_pass4(const double2 *in, double2 *out, int n, int Ns, int tstride,
                                              bool inverse, const double2 *tw, int Mh, int lane)
{
    const int quarter = n >> 2;
    for (int j = lane; j < quarter; j += 32) {
        const int k = j & (Ns - 1);
        const int m = k * tstride;
        const double2 a = in[j];
        const double2 b = cmul(fin_tw(tw, m, Mh, inverse), in[j + quarter]);
        const double2 c = cmul(fin_tw(tw, 2 * m, Mh, inverse), in[j + 2 * quarter]);
        const double2 d = cmul(fin_tw(tw, 3 * m, Mh, inverse), in[j + 3 * quarter]);
        const double2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = csub(b, d);
        // -i (b - d) forward, +i (b - d) inverse
        const double2 r3 = inverse ? make_double2(-s3.y, s3.x) : make_double2(s3.y, -s3.x);
        const int j0 = ((j - k) << 2) + k;
        out[j0] = cadd(s0, s2);
        out[j0 + Ns] = cadd(s1, r3);
        out[j0 + 2 * Ns] = csub(s0, s2);
        out[j0 + 3 * Ns] = csub(s1, r3);
    }
}

// n-point FFT (n a power of two >= 4) by radix-4 passes and one radix-2 pass if needed; returns
// the buffer that holds the result.
__device__ __forceinline__ double2 *fin_fft(double2 *src, double2 *dst, int n, int M, bool inverse,
                                            const double2 *tw, int lane)
{
    int Ns = 1;
    for (; Ns * 4 <= n; Ns <<= 2) {
        fin_fft_pass4(src, dst, n, Ns, M / (4 * Ns), inverse, tw, M >> 1, lane);
        __syncwarp();
        double2 *tmp = src; src = dst; dst = tmp;
    }
    if (Ns < n) {
        fin_fft_pass(src, dst, n, Ns, M / (2 * Ns), inverse, tw, lane);
        __syncwarp();
        double2 *tmp = src; src = dst; dst = tmp;
    }
    return src;
}

// usb / lsb staging layout: output k of lane segment g = k >> lsh sits at g*Ls + ((k + g) mod Ls), a
// rotation inside its own aligned segment -- conflict-free both for the lane <-> block writes of
// phase 3 and for the lane <-> segment passes, and it never leaves the 32-output tile of k (Ls <= 32)
__device__ __forceinline__ int fin_ssb_at(int k, int lsh, int Ls)
{
    const int g = k >> lsh;
    return (g << lsh) | ((k + g) & (Ls - 1));
}

template <int ENC, int OUT>
__global__ void __launch_bounds__(32 * FIN_WARPS, 2)
k_finish(const __grid_constant__ DevPlan pl, const __grid_constant__ Scratch sc, const uint8_t *__restrict__ raw,
         double *__restrict__ out, int nchunks, int keep_y)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int M = pl.M, nt = pl.ntiles, edge = pl.edge, R = pl.R, h = M >> 1, n2 = M >> 2;
    const bool iq = pl.correct_iq != 0;

    double2 *tw = reinterpret_cast<double2 *>(smem_raw);                 // exp(-2 pi i k / M), k < M/2
    double2 *pk = tw + h;                                                // p_i^k, [edge+1][8]
    for (int k = threadIdx.x; k < h; k += blockDim.x) tw[k] = pl.tw[k];
    for (int k = threadIdx.x; k < (edge + 1) * 8; k += blockDim.x) pk[k] = pl.pk[k];
    // row tables: resident in shared memory when the bank has one row (the L1 copies are evicted
    // by the streaming ypart / agg reads), read from global memory per item otherwise
    double2 *tbT1 = pk + (edge + 1) * 8, *tbPsi = tbT1 + nt, *tbPt = tbPsi + 48, *tbEh = tbPt + nt * 8,
            *tbEe = tbEh + 32, *tbPy = tbEe + 32;
    if (R == 1) {
        for (int k = threadIdx.x; k < nt; k += blockDim.x) tbT1[k] = pl.T1[k];
        // tbPsi: per-mode IQ constants of the row: alpha, alphaT | 1/beta, 1/betaT | beta, betaT (lanes 0..7 / 8..15)
        for (int k = threadIdx.x; k < 16; k += blockDim.x) {
            tbPsi[k] = k < 8 ? pl.alpha[k] : pl.alphaT[k - 8];
            tbPsi[16 + k] = k < 8 ? pl.binv[k] : pl.binvT[k - 8];
            tbPsi[32 + k] = k < 8 ? pl.beta[k] : pl.betaT[k - 8];
        }
        for (int k = threadIdx.x; k < nt * 8; k += blockDim.x) tbPt[k] = pl.Pt[k];
        for (int k = threadIdx.x; k <= edge; k += blockDim.x) { tbEh[k] = pl.Ehead[k]; tbEe[k] = pl.Eend[k]; }
        for (int k = threadIdx.x; k < 64; k += blockDim.x) tbPy[k] = pl.psiY[k];
    }
    unsigned char *wb = smem_raw + (size_t)(h + (edge + 1) * 8 + nt + 48 + nt * 8 + 32 + 32 + 64) * sizeof(double2) +
                        (size_t)warp * finish_warp_bytes(M);
    double2 *carry = reinterpret_cast<double2 *>(wb);
    double2 *fa = carry + (size_t)(nt + 1) * 16, *fb = carry;            // fb: only after the outputs (carry dead)
    // phase-1 scratch overlays fa and the (not yet written) zrow: addv [nt][16], then seqA, seqB
    double2 *addv = fa;                                                  // dead before the FFT buffers are written
    double2 *seqA = fa + (size_t)nt * 16, *seqB = seqA + 32;             // dead before zrow is written
    double *zrow = reinterpret_cast<double *>(fa + n2);
    __syncthreads();

    // lane-invariant tables: this lane's block position l = lane inside every tile
    // (the filter is real: poles 4..7 are the conjugates of 0..3 and so are their weights, hence
    // sum_i c_i w_i = 2 Re(c_i Wr_i) + 2j Re(c_i Wi_i) over i < 4 with the modal states of the real and
    // imaginary input streams Wr = (w_i + conj w_{i+4}) / 2, Wi = (w_i - conj w_{i+4}) / 2j: half the FMAs)
    double2 rw[4], rt[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        rw[i] = cscale(2.0, pl.RW[(size_t)lane * 8 + i]);
        rt[i] = cscale(2.0, pl.RT[(size_t)(SDRB_TB - lane) * 8 + i]);
    }
    const int i8 = lane & 7, grp = (lane >> 3) & 1, sub = lane >> 3;
    const double2 p_i = pl.p[i8], P32 = pl.Ppow[(size_t)SDRB_TB * 8 + i8];
    const int Ls = pl.sos_Lseg, lsh = Ls > 0 ? 31 - __clz(Ls) : 31;   // no output SOS (re/im): no padding
    const int dchunk = (edge + 3) >> 2;                                  // dot-product terms per lane group
    const double lamn = pl.lam_pw[lane], mun = pl.mu_pw[min(32, max(0, edge + 1 - lane))];

    const int gw = blockIdx.x * FIN_WARPS + warp, nw = gridDim.x * FIN_WARPS;
    int nit = -1;
    for (int item = gw; item < nchunks * R; item += nw) {
        nit++;
        FIN_DBG(0);
        const int chunk = item / R, r = item - chunk * R;
        const uint8_t *rawc = raw + (size_t)chunk * pl.N * pl.sb;
        const double2 *aggr = sc.agg + ((size_t)chunk * R + r) * nt * 16;
        const double2 *T1r = R == 1 ? tbT1 : pl.T1 + (size_t)r * nt;
        const double2 *ypr = sc.ypart + ((size_t)chunk * R + r) * pl.Mf;

        // ---------------------------------------------------------------- 1a. loads
        double2 xh = make_double2(0.0, 0.0), xe = make_double2(0.0, 0.0);
        if (lane <= edge) {
            xh = decode_sample<ENC>(pl, rawc, lane);
            xe = decode_sample<ENC>(pl, rawc, (long)pl.ws + lane);
        }
        // offsets at the tile starts from the chunk-start offset and the tile aggregates of the
        // front end: lane t keeps the offset entering tile t (shuffled out where needed); oE = the
        // offset at the end of the chunk
        double2 offr = make_double2(0.0, 0.0), oE = offr;
        if (iq) {
            const TileOffsets to = tile_offsets(pl, sc.tile_agg + (size_t)chunk * nt, sc.start[chunk], lane);
            offr = to.in;
            oE = to.end;
        }
        {   // the next item's inputs start their way into L2 now
            const int nitem = item + nw;
            if (nitem < nchunks * R) {
                const int nchunk = nitem / R, nr = nitem - nchunk * R;
                const char *py = reinterpret_cast<const char *>(sc.ypart + ((size_t)nchunk * R + nr) * pl.Mf);
                const char *pa = reinterpret_cast<const char *>(sc.agg + ((size_t)nchunk * R + nr) * nt * 16);
                for (int o = lane * 128; o < M * 16; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(py + o));
                for (int o = lane * 128; o < nt * 256; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pa + o));
                if (lane < 2) {
                    const uint8_t *pr = raw + (size_t)nchunk * pl.N * pl.sb + (lane ? (size_t)pl.ws * pl.sb : 0);
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(pr));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(pr + 128));
                }
            }
        }
        for (int i0 = 0; i0 < nt * 16; i0 += 8 * 32) {
            double2 av[8];
#pragma unroll
            for (int u = 0; u < 8; u++)
                av[u] = (i0 + u * 32 + lane < nt * 16) ? aggr[i0 + u * 32 + lane] : make_double2(0.0, 0.0);
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int idx = i0 + u * 32 + lane, t = min(idx >> 4, nt - 1), m = idx & 15;
                // the aggregates are sums of the UNcorrected samples: no offset term here (3.3)
                if (idx < nt * 16) addv[idx] = cmul(T1r[min(t, nt - 1)], av[u]);
                (void)m;
            }
        }
        FIN_DBG(1);
        // ---------------------------------------------------------------- 1b. IQ correction
        // read_file.py:72-77 is the linear recurrence off' = lam off + L z; lane <-> sample.  Head:
        // off_n = lam^n off_0 + L sum_{i<n} lam^(n-1-i) z_i (scan upwards).  End window, from the
        // offset at q*Mf backwards: off_n = mu^m off_E - L mu sum_{i>=n} mu^(i-n) z_i, mu = 1/lam.
        if (iq) {
            const double2 o0 = shfl_c(offr, 0);
            double2 S = xh, B = xe;
#pragma unroll
            for (int lv = 0; lv < 5; lv++) {
                const double2 tu = shfl_up_c(S, 1 << lv);
                const double2 td = make_double2(__shfl_down_sync(0xffffffffu, B.x, 1 << lv), __shfl_down_sync(0xffffffffu, B.y, 1 << lv));
                if (lane >= (1 << lv)) { S.x = fma(pl.lam_pw[1 << lv], tu.x, S.x); S.y = fma(pl.lam_pw[1 << lv], tu.y, S.y); }
                if (lane + (1 << lv) < 32) { B.x = fma(pl.mu_pw[1 << lv], td.x, B.x); B.y = fma(pl.mu_pw[1 << lv], td.y, B.y); }
            }
            double2 Sx = shfl_up_c(S, 1);
            if (lane == 0) Sx = make_double2(0.0, 0.0);
            xh.x -= fma(lamn, o0.x, pl.Liq * Sx.x); xh.y -= fma(lamn, o0.y, pl.Liq * Sx.y);
            const double lm = pl.Liq * pl.mu_pw[1];
            xe.x -= fma(mun, oE.x, -lm * B.x); xe.y -= fma(mun, oE.y, -lm * B.y);
        }
        FIN_DBG(2);
        // ---------------------------------------------------------------- 1c. NCO, odd extensions
        if (lane <= edge) {
            xh = cmul(xh, R == 1 ? tbEh[lane] : pl.Ehead[(size_t)r * (edge + 1) + lane]);
            xe = cmul(xe, R == 1 ? tbEe[lane] : pl.Eend[(size_t)r * pl.nend + lane]);
        }
        {
            const double2 x0 = shfl_c(xh, 0), xN1 = shfl_c(xe, edge);
            const double2 ha = shfl_c(xh, max(0, edge - lane)), eb = shfl_c(xe, max(0, edge - 1 - lane));
            if (lane < edge) {
                seqA[lane] = make_double2(fma(2.0, x0.x, -ha.x), fma(2.0, x0.y, -ha.y));       // head extension
                seqB[lane] = make_double2(fma(2.0, xN1.x, -eb.x), fma(2.0, xN1.y, -eb.y));     // tail extension
            }
        }
        __syncwarp();
        FIN_DBG(3);
        // ---------------------------------------------------------------- 1d. head / tail states
        // closed forms of the serial recurrences: w(edge) = p^edge zhat ext0 + sum_j p^(edge-1-j) ext_j,
        // T(end) = sum_k p^k tail_k, and the tail-driven part of w(L-2); lane = (pole, quarter of j)
        double2 accA = make_double2(0.0, 0.0), accB = accA, accC = accA;
        {
            const int j0 = sub * dchunk, j1 = min(edge, j0 + dchunk);
            for (int j = j0; j < j1; j++) {
                const double2 a = seqA[j], b = seqB[j];
                accA = cfma(pk[(edge - 1 - j) * 8 + i8], a, accA);
                accB = cfma(pk[j * 8 + i8], b, accB);
                if (j <= edge - 2) accC = cfma(pk[(edge - 2 - j) * 8 + i8], b, accC);
            }
#pragma unroll
            for (int sft = 8; sft < 32; sft <<= 1) {
                accA = cadd(accA, shfl_xor_c(accA, sft));
                accB = cadd(accB, shfl_xor_c(accB, sft));
                accC = cadd(accC, shfl_xor_c(accC, sft));
            }
            accA = cfma(pk[edge * 8 + i8], cmul(pl.zhat[i8], seqA[0]), accA);
        }
        FIN_DBG(4);
        // ---------------------------------------------------------------- 1e. carries across tiles
        // lanes 0..7: forward modal states (Win[t] = state entering tile t); lanes 8..15: anticausal
        // states (Tn[t] = state entering tile t from above)
        // in the frame of the uncorrected samples (3.3): W~ = (w + alpha s) / beta at n = 0,
        // T~ = (T + alphaT s) / betaT at n = q*Mf, s = off e^{jwn}; stored pre-scaled by beta / betaT
        double2 st = grp ? accB : accA;
        double2 qal = make_double2(0.0, 0.0), qbe = make_double2(1.0, 0.0), sE = qal;
        const double2 o0c = shfl_c(offr, 0);
        if (iq) {
            const int mi = grp * 8 + i8;
            qal = R == 1 ? tbPsi[mi] : (grp ? pl.alphaT : pl.alpha)[(size_t)r * 8 + i8];
            const double2 qbi = R == 1 ? tbPsi[16 + mi] : (grp ? pl.binvT : pl.binv)[(size_t)r * 8 + i8];
            qbe = (grp ? pl.betaT : pl.beta)[(size_t)r * 8 + i8];
            sE = cmul(oE, pl.phE[r]);
            st = cmul(cfma(qal, grp ? sE : o0c, st), qbi);
        }
        // (the chain itself stays in the frame of the uncorrected samples; beta / betaT are applied
        // when the carries are turned into real / imaginary stream states below)
        if (lane >= 8 && lane < 16) carry[(size_t)nt * 16 + 8 + i8] = st;
        for (int tt = 0; tt < nt; tt++) {
            const int t = grp ? nt - 1 - tt : tt;
            if (lane < 8) carry[(size_t)t * 16 + i8] = st;
            st = cfma(P32, st, addv[t * 16 + grp * 8 + i8]);
            if (lane >= 8 && lane < 16) carry[(size_t)t * 16 + 8 + i8] = st;
        }
        if (lane < 8) carry[(size_t)nt * 16 + i8] = st;
        if (iq) st = csub(cmul(qbe, st), cmul(qal, sE));    // lanes 0..7: the TRUE forward state at q*Mf
        FIN_DBG(5);
        // ---------------------------------------------------------------- 1f. boundary vector zeta
        {
            const double2 Wn = shfl_c(st, i8);                              // forward state at n = edge + q*Mf
            const double2 last = seqB[edge - 1];
            const double2 wL1 = cfma(pk[(edge - 1) * 8 + i8], Wn, accC);
            const double2 wL = cfma(p_i, wL1, last);
            double2 part = cmul(pl.c[i8], wL1);
            for (int sft = 1; sft < 8; sft <<= 1) part = cadd(part, shfl_xor_c(part, sft));
            const double2 yfL1 = make_double2(fma(pl.d, last.x, part.x), fma(pl.d, last.y, part.y));
            double2 za = cmul(pl.zhat[i8], yfL1), zb = make_double2(0.0, 0.0);
#pragma unroll
            for (int l = 0; l < 8; l += 2) {
                za = csub(za, cmul(pl.xi[i8 * 8 + l], shfl_c(wL, l)));
                zb = csub(zb, cmul(pl.xi[i8 * 8 + l + 1], shfl_c(wL, l + 1)));
            }
            // sosfiltfilt's boundary term c_i p_i^(L-1-n) zeta_i is an anticausal modal response:
            // it rides on the backward carries as X_i = p_i^edge / kappa_i zeta_i at n = edge + q*Mf
            double2 X = cmul(pl.bx[i8], cadd(za, zb));
            if (iq) X = cmul(X, R == 1 ? tbPsi[24 + i8] : pl.binvT[(size_t)r * 8 + i8]);   // into the T~ frame
            __syncwarp();
            for (int t = sub; t < nt; t += 4) {
                double2 *Tn = carry + (size_t)(t + 1) * 16 + 8 + i8;
                *Tn = cfma((R == 1 ? tbPt : pl.Pt)[(size_t)(nt - 1 - t) * 8 + i8], X, *Tn);
            }
        }
        __syncwarp();
        // carries -> states of the real / imaginary input streams (slots i and i + 4 of each group)
        for (int idx = lane; idx < (nt + 1) * 8; idx += 32) {
            double2 *c = carry + (size_t)(idx >> 2) * 8 + (idx & 3);       // group = (tile, direction)
            double2 a = c[0], b = c[4];
            if (iq) {                                                       // beta W~, betaT T~
                const int d8 = ((idx >> 2) & 1) * 8 + (idx & 3);
                const double2 b0 = R == 1 ? tbPsi[32 + d8] : (((idx >> 2) & 1) ? pl.betaT : pl.beta)[(size_t)r * 8 + (idx & 3)];
                const double2 b4 = R == 1 ? tbPsi[32 + d8 + 4] : (((idx >> 2) & 1) ? pl.betaT : pl.beta)[(size_t)r * 8 + (idx & 3) + 4];
                a = cmul(b0, a); b = cmul(b4, b);
            }
            b = cconj(b);
            c[0] = make_double2(0.5 * (a.x + b.x), 0.5 * (a.y + b.y));
            c[4] = make_double2(0.5 * (a.y - b.y), -0.5 * (a.x - b.x));
        }
        __syncwarp();
        FIN_DBG(6);
        // ---------------------------------------------------------------- 2+3a. outputs, lane <-> block
        // y[k] = T1 (ypart - off psi) + sum_i rho_i P_i^l Win_i + rho_i/p_i P_i^(32-l) Tn_i (+ boundary),
        // two tiles per round; fm forms the pair phases in registers (even lanes take tile t0's
        // pairs, odd lanes tile t1's), the other modes go straight to the output row
        {
            double2 *yg = sc.y + ((size_t)chunk * R + r) * M;
            const double2 psi0 = R == 1 ? tbPy[lane] : pl.psiY[((size_t)0 * R + r) * SDRB_TB + lane];
            const double2 psi1 = R == 1 ? tbPy[32 + lane] : pl.psiY[((size_t)1 * R + r) * SDRB_TB + lane];
            double *ph = reinterpret_cast<double *>(fa);
            // ypart is fetched two rounds (four tiles) ahead of its use
            double2 yq[4];
#pragma unroll
            for (int u = 0; u < 4; u++) yq[u] = u < nt ? ypr[u * SDRB_TB + lane] : make_double2(0.0, 0.0);
            for (int t0 = 0; t0 < nt; t0 += 2) {
                double2 yv[2];
                const double2 yin0 = yq[0], yin1 = yq[1];
                yq[0] = yq[2]; yq[1] = yq[3];
                if (t0 + 4 < nt) { yq[2] = ypr[(t0 + 4) * SDRB_TB + lane]; yq[3] = ypr[(t0 + 5) * SDRB_TB + lane]; }
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int t = t0 + u, k = t * SDRB_TB + lane;
                    double2 v = u ? yin1 : yin0;
                    if (iq) {
                        const double2 o = shfl_c(offr, t);
                        v = cfma(make_double2(-o.x, -o.y), (t == nt - 1) ? psi1 : psi0, v);
                    }
                    v = cmul(T1r[t], v);
                    const double2 *Win = carry + (size_t)t * 16, *Tn = carry + (size_t)(t + 1) * 16 + 8;
                    double2 a1 = make_double2(0.0, 0.0);
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        v.x = fma(rw[i].x, Win[i].x, fma(-rw[i].y, Win[i].y, v.x));
                        v.y = fma(rw[i].x, Win[i + 4].x, fma(-rw[i].y, Win[i + 4].y, v.y));
                        a1.x = fma(rt[i].x, Tn[i].x, fma(-rt[i].y, Tn[i].y, a1.x));
                        a1.y = fma(rt[i].x, Tn[i + 4].x, fma(-rt[i].y, Tn[i + 4].y, a1.y));
                    }
                    v = cadd(v, a1);
                    if (keep_y) yg[k] = v;
                    yv[u] = v;
                }
                if constexpr (OUT == OUT_IQ) {
                    // 16 contiguous bytes per lane, 512 per warp and tile: no trip through zrow
                    double2 *o2 = reinterpret_cast<double2 *>(out + ((size_t)r * nchunks + chunk) * pl.W);
#pragma unroll
                    for (int u = 0; u < 2; u++) frame_store(o2 + (t0 + u) * SDRB_TB + lane, yv[u], pl.be_out);
                } else if constexpr (OUT == OUT_SSB) {
                    // Re y -> zrow; Im y -> the carry rows t0, t0+1, dead once every lane has read them
                    __syncwarp();
                    double *zim = reinterpret_cast<double *>(carry);
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        const int a = fin_ssb_at((t0 + u) * SDRB_TB + lane, lsh, Ls);
                        zrow[a] = yv[u].x;
                        zim[a] = yv[u].y;
                    }
                } else if (pl.demod == 0) {
                    const bool odd = lane & 1;
                    const double2 snd = odd ? yv[0] : yv[1];
                    const double2 rcv = shfl_xor_c(snd, 1);
                    const double v = pair_phase(odd ? rcv : yv[0], odd ? yv[1] : rcv);
                    const int i = 16 * (t0 + (odd ? 1 : 0)) + (lane >> 1);
                    ph[i] = v;
                    zrow[2 * i + ((2 * i) >> lsh)] = v;
                } else {
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        const int k = (t0 + u) * SDRB_TB + lane;
                        zrow[k + (k >> lsh)] = demod_scalar(yv[u], pl.demod);
                    }
                }
            }
        }
        __syncwarp();
        FIN_DBG(7);
        // ---------------------------------------------------------------- 3b. fm: 2x interpolation
        if (OUT == OUT_REAL && pl.demod == 0) {
            // even outputs of scipy.signal.resample(ph, 2h) are the phases themselves (already in
            // zrow), the odd ones come from the half-sample-shifted spectrum.  Forward FFT of
            // z[m] = ph[2m] + i ph[2m+1], n2 = h/2 points
            double2 *src = fin_fft(fa, fb, n2, M, false, tw, lane);
            double2 *dst = src == fa ? fb : fa;
            // spectrum of the real row X[k] (k <= h/2) from Z, times the half-sample shift
            // H[k] = exp(i pi k / h), re-packed for the half-length inverse transform
            for (int k = lane; k <= (n2 >> 1); k += 32) {
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
            __syncwarp();
            src = fin_fft(dst, src, n2, M, true, tw, lane);
            const double sc1 = 1.0 / (double)h;
            for (int m = lane; m < n2; m += 32) {
                const double2 v = src[m];
                const int k1 = 4 * m + 1, k3 = 4 * m + 3;
                zrow[k1 + (k1 >> lsh)] = v.x * sc1;
                zrow[k3 + (k3 >> lsh)] = v.y * sc1;
            }
            __syncwarp();
        }
        FIN_DBG(8);
        // ---------------------------------------------------------------- 4. output filter
        // fm / am: the low-pass over the padded row (segment g at g (Ls + 1)); usb / lsb: the band-pass
        // over y staged at fin_ssb_at, Re in zrow and Im in the carry rows; the kept output -> zrow
        if constexpr (OUT != OUT_IQ) {
            if (OUT == OUT_SSB || pl.nsec_out > 0) {
                const double *zim = reinterpret_cast<const double *>(carry);
                double *zs = zrow + (OUT == OUT_SSB ? 0 : (size_t)lane * (Ls + 1));
                auto at = [&](int j) { return OUT == OUT_SSB ? lane * Ls + ((j + lane) & (Ls - 1)) : j; };
                std::conditional_t<OUT == OUT_SSB, double2, double> st[4];
                sos_segments(
                    pl, 2, lane * Ls, Ls, lane,
                    [&](int j) {
                        if constexpr (OUT == OUT_SSB) return make_double2(zs[at(j)], zim[at(j)]);
                        else return zs[at(j)];
                    },
                    [&](int j) -> double & { return zs[at(j)]; }, st);
                __syncwarp();
            }
        }
        FIN_DBG(9);
        // ---------------------------------------------------------------- 5. framing
        if constexpr (OUT != OUT_IQ) {
            double *o = out + ((size_t)r * nchunks + chunk) * M;
            for (int k = lane; k < M; k += 32)
                frame_store(o + k, zrow[OUT == OUT_SSB ? fin_ssb_at(k, lsh, Ls) : k + (k >> lsh)], pl.be_out);
            __syncwarp();
        }
        FIN_DBG(10);
    }
}
