// sdrb_finish.cuh -- k_finish: everything after the block front end, one warp per (chunk, row).
//
//   1. chunk boundaries: IQ-corrected, NCO-shifted head and end-window samples; sosfiltfilt's odd
//      extension and zi start-up (head), the tail extension (end), the boundary vector zeta -- the
//      chunk-boundary routines of sdrb_kernels.cuh, which k_fixup and the seamless kernels run too
//   2. carries of the 8 forward / 8 anticausal modal states across the tiles of the chunk
//   3. decimated outputs y[k] = partial output of the front end + carry-in response (+ boundary)
//   4. demodulation: fm (pair phase, 2x trigonometric interpolation: sdrb_fft.cuh's fm_interp2x on
//      the warp) | am | re | im; the iq instance (OUT_IQ) stores y straight from registers
//      instead, (Re, Im) per output, and skips 3b-5
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
// emu_demod) is the numpy twin.
#pragma once
#include "sdrb_fft.cuh"
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
    const double2 P32 = pl.Ppow[(size_t)SDRB_TB * 8 + i8];
    const int Ls = pl.sos_Lseg, lsh = Ls > 0 ? 31 - __clz(Ls) : 31;   // no output SOS (re/im): no padding

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
        // ---------------------------------------------------------------- 1b. IQ correction, NCO
        // head forward from the chunk-start offset; end window (nend = edge + 1 samples: rem = 0)
        // backward from the offset at q*Mf
        const double2 o0 = shfl_c(offr, 0);
        {
            double2 Eh = make_double2(0.0, 0.0), Ee = Eh;
            if (lane <= edge) {
                Eh = R == 1 ? tbEh[lane] : pl.Ehead[(size_t)r * (edge + 1) + lane];
                Ee = R == 1 ? tbEe[lane] : pl.Eend[(size_t)r * pl.nend + lane];
            }
            xh = edge_correct(pl, xh, o0, edge + 1, 0, Eh, lane).x;
            xe = edge_correct(pl, xe, oE, edge + 1, edge + 1, Ee, lane).x;
        }
        FIN_DBG(2);
        // ---------------------------------------------------------------- 1c. odd extensions
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
        const BoundarySums bs = boundary_sums(pl, pk, seqA, edge, seqB, edge, lane);
        FIN_DBG(4);
        // ---------------------------------------------------------------- 1e. carries across tiles
        // lanes 0..7: forward modal states (Win[t] = state entering tile t); lanes 8..15: anticausal
        // states (Tn[t] = state entering tile t from above)
        // in the frame of the uncorrected samples (3.3): W~ = (w + alpha s) / beta at n = 0,
        // T~ = (T + alphaT s) / betaT at n = q*Mf, s = off e^{jwn}; stored pre-scaled by beta / betaT
        double2 st = grp ? bs.B : bs.A;
        double2 qal = make_double2(0.0, 0.0), qbe = make_double2(1.0, 0.0), sE = qal;
        if (iq) {
            const int mi = grp * 8 + i8;
            qal = R == 1 ? tbPsi[mi] : (grp ? pl.alphaT : pl.alpha)[(size_t)r * 8 + i8];
            const double2 qbi = R == 1 ? tbPsi[16 + mi] : (grp ? pl.binvT : pl.binv)[(size_t)r * 8 + i8];
            qbe = (grp ? pl.betaT : pl.beta)[(size_t)r * 8 + i8];
            sE = cmul(oE, pl.phE[r]);
            st = cmul(cfma(qal, grp ? sE : o0, st), qbi);
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
            // from the forward state at n = edge + q*Mf: sosfiltfilt's boundary term c_i p_i^(L-1-n)
            // zeta_i is an anticausal modal response: it rides on the backward carries as
            // X_i = p_i^edge / kappa_i zeta_i at n = edge + q*Mf
            double2 X = cmul(pl.bx[i8], boundary_zeta(pl, pk, seqB, edge, shfl_c(st, i8), bs.C, lane));
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
            // zrow), the odd ones come from the half-sample-shifted spectrum
            fm_interp2x(fa, fb, M, tw, WarpGroup{lane}, [&](int k, double v) { zrow[k + (k >> lsh)] = v; });
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
