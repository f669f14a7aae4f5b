// sdrb_kernels.cuh -- the sm_100a kernels of the demodulation chain.
//
//   k_main     raw tile -> shared memory; run-wise IQ correction, NCO and the even/odd block sums
//              on the FP64 tensor pipe (DMMA.8x8x4), all from registers; tile-local modal scans
//              -> partial outputs + tile aggregates
//   k_iqgain / k_iqscan_c / k_iqtiles   IQ-corrector offset at every tile start, carried across
//              chunks and calls: chunk gains (warp <-> chunk), the chunk scan (one CTA), the tile
//              offsets (warp <-> chunk; k_finish derives them itself); tile_offsets is the one
//              tile-offset routine of all three and k_finish
//   k_iqchunk  chunk gains straight from the raw bytes (time-segment sharding)
//   k_fixup    chunk boundary (head, end window, boundary sums and zeta: the chunk-boundary routines
//              of k_finish and the seamless kernels too), cross-tile carries -> decimated complex y
//   k_demod    fm (pair phase + 2x FFT interpolation) | am | re | im, output SOS, framing; iq: y
//              itself framed as (Re, Im) pairs; usb / lsb: the complex band-pass on y, its real part
//              framed.  The demodulator scalars and the output SOS (32 lane segments, lane scan,
//              per-output correction) are sdrb_outstage.cuh's, shared with k_finish and seamless mode
//
// Reference behaviour being reproduced: src/misc/read_file.py:100-103 (decode, normalise, IQ
// correction), src/dsp/demodulation.py:71-79 (NCO), src/dsp/dsp_processor.py:147 (scipy
// decimate), demodulation.py:25-68, dsp_processor.py:32-36,149,162, vfo_processor.py:84.
// tests/emulator.py is the numpy twin of these kernels (same tables, same decomposition).
#pragma once
#include "sdrb_device.cuh"
#include "sdrb_fft.cuh"
#include "sdrb_outstage.cuh"

// Scratch written by k_main / read by k_fixup, per batch of chunks.
struct Scratch {
    double2 *ypart;     // [nch][R][Mf]
    double2 *agg;       // [nch][R][ntiles][16]   0..7 Wout, 8..15 Tin
    double2 *tile_agg;  // [nch][ntiles]
    double2 *off_tile;  // [nch][ntiles+1]
    double2 *gain;      // [nch] offset gained over a chunk from zero
    double2 *start;     // [nch] offset at the chunk start
    double2 *carry;     // [nch][R][ntiles+1][16] 0..7 Win[t], 8..15 Tn[t]
    double2 *y;         // [nch][R][M]
    double2 *iq_state;  // [1] offset before the batch (in) / after it (out)
    double2 *fftbuf;    // [nch*R] k_demod row scratch of demod_smem_bytes(M) when it does not fit shared memory
    unsigned long long *dbg;  // optional k_tc timeline (SDRB_TC_DEBUG): [64 tiles][16 events] clock64 of CTA 0
    double2 *x0;        // optional [nch][R][Mf]: first raw sample of every block as the tensor-core
                        // front end sees it (exact integers; sdrb_keep_x0, parity tests)
};

// Shared-memory carve-up of k_main (host mirrors this in sdrb_api.cu).
// A raw tile is kept in the order the DMMA fragments consume it: slot (s, g, lane) holds the two
// raw samples lane = (block 8g + (lane>>2), pair kq*RL + s) multiplies in step s of group g --
// sample j and its mirror q-1-j -- side by side, so a lane fetches a pair with ONE shared-memory
// load of 2*sb bytes, conflict-free, and no address arithmetic on the row.  Planes of one s are
// 256*sb bytes apart plus 16 bytes of skew (the staging stores of a warp walk along s).
__host__ __device__ inline size_t main_plane_bytes(int sb) { return (size_t)256 * sb + 16; }
__host__ __device__ inline size_t main_tile_bytes(int RL, int sb)
{
    return (size_t)RL * main_plane_bytes(sb) + 2 * SDRB_TB * sizeof(double2);   // pairs + cl[32], blkagg[32]
}
__host__ __device__ inline size_t main_warp_bytes()
{
    return (size_t)32 * SDRB_XSTRIDE * sizeof(double) + SDRB_TB * sizeof(double2);  // xb + x0s
}

// Raw tiles of one CTA -> shared memory in fragment order, one word of type T per sample: every
// warp takes four block rows at a time and issues their loads together (rows past the chunk's
// last block are zero).
// Stored byte order -> the GPU's, one raw sample (two items) at a time: done once when the tile is
// staged, not once per row of the bank.
__device__ __forceinline__ uint16_t swap_items(uint16_t v) { return v; }
__device__ __forceinline__ uint32_t swap_items(uint32_t v) { return __byte_perm(v, 0, 0x2301); }
__device__ __forceinline__ uint2 swap_items(uint2 v) { return make_uint2(__byte_perm(v.x, 0, 0x0123), __byte_perm(v.y, 0, 0x0123)); }
__device__ __forceinline__ uint4 swap_items(uint4 v)
{
    return make_uint4(__byte_perm(v.y, 0, 0x0123), __byte_perm(v.x, 0, 0x0123), __byte_perm(v.w, 0, 0x0123), __byte_perm(v.z, 0, 0x0123));
}

template <typename T>
__device__ __forceinline__ void stage_pairs(unsigned char *tiles, size_t tileb, const uint8_t *rawc, int t0, int ntl,
                                            int ntiles, int cnt_last, int q, int Hq, int RL, int swap, int warp, int W, int lane)
{
    const int total = ntl * SDRB_TB;
    const size_t plane = main_plane_bytes((int)sizeof(T));
    for (int r0 = warp * 4; r0 < total; r0 += W * 4) {
        const int tl = r0 >> 5, row0 = r0 & 31, t = t0 + tl;          // four rows never straddle a tile
        const int cnt = (t == ntiles - 1) ? cnt_last : SDRB_TB;
        const T *src = reinterpret_cast<const T *>(rawc) + ((size_t)t * SDRB_TB + row0) * q;
        unsigned char *tb = tiles + (size_t)tl * tileb;
        for (int col = lane; col < q; col += 32) {
            const int slot = col < Hq ? 0 : 1, jj = slot ? q - 1 - col : col;
            const int kq = jj / RL, sp = jj - kq * RL;
            T v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) v[u] = (row0 + u < cnt) ? src[(size_t)u * q + col] : T{};
            if (swap) {
#pragma unroll
                for (int u = 0; u < 4; u++) v[u] = swap_items(v[u]);
            }
            T *dst = reinterpret_cast<T *>(tb + (size_t)sp * plane) + ((size_t)(row0 >> 3) * 32 + (row0 & 7) * 4 + kq) * 2 + slot;
#pragma unroll
            for (int u = 0; u < 4; u++) dst[u * 8] = v[u];           // next block row: lane slot + 4 = 8 words on
        }
    }
    // slots no sample lands in -- pairs Hq .. 4 RL - 1 and the mirror of an odd block's middle
    // sample -- are zero: their modal coefficients are zero, so the data only has to be finite
    const int nempty = 2 * (4 * RL - Hq) + (q & 1);
    for (int idx = warp * 32 + lane; idx < nempty * SDRB_TB * ntl; idx += W * 32) {
        const int b = idx & 31, k = (idx >> 5) % nempty, tl = (idx >> 5) / nempty;
        const int jj = k < 2 * (4 * RL - Hq) ? Hq + (k >> 1) : Hq - 1, slot = k < 2 * (4 * RL - Hq) ? (k & 1) : 1;
        const int kq = jj / RL, sp = jj - kq * RL;
        reinterpret_cast<T *>(tiles + (size_t)tl * tileb + (size_t)sp * plane)[((size_t)(b >> 3) * 32 + (b & 7) * 4 + kq) * 2 + slot] = T{};
    }
}

// The pair of slot (s, g, lane) -> two complex doubles (decode of read_file.py:100-101 from
// registers; the byte order was fixed when the tile was staged).
template <int ENC>
__device__ __forceinline__ void load_pair(const DevPlan &pl, const unsigned char *plane_s, int g, int lane, double2 &za, double2 &zb)
{
    const int idx = g * 32 + lane;
    if (ENC == ENC_b || ENC == ENC_B) {
        const uint32_t v = reinterpret_cast<const uint32_t *>(plane_s)[idx];
        if (ENC == ENC_b) {
            za = make_double2((double)(int8_t)(v & 0xff), (double)(int8_t)((v >> 8) & 0xff));
            zb = make_double2((double)(int8_t)((v >> 16) & 0xff), (double)(int8_t)(v >> 24));
        } else {
            za = make_double2((double)(v & 0xff), (double)((v >> 8) & 0xff));
            zb = make_double2((double)((v >> 16) & 0xff), (double)(v >> 24));
        }
    } else if (ENC == ENC_h || ENC == ENC_H) {
        const uint2 v = reinterpret_cast<const uint2 *>(plane_s)[idx];
        if (ENC == ENC_h) {
            za = make_double2((double)(int16_t)(v.x & 0xffff), (double)(int16_t)(v.x >> 16));
            zb = make_double2((double)(int16_t)(v.y & 0xffff), (double)(int16_t)(v.y >> 16));
        } else {
            za = make_double2((double)(v.x & 0xffff), (double)(v.x >> 16));
            zb = make_double2((double)(v.y & 0xffff), (double)(v.y >> 16));
        }
    } else if (ENC == ENC_i || ENC == ENC_I || ENC == ENC_f) {
        const uint4 v = reinterpret_cast<const uint4 *>(plane_s)[idx];
        if (ENC == ENC_i) {
            za = make_double2((double)(int32_t)v.x, (double)(int32_t)v.y); zb = make_double2((double)(int32_t)v.z, (double)(int32_t)v.w);
        } else if (ENC == ENC_I) {
            za = make_double2((double)v.x, (double)v.y); zb = make_double2((double)v.z, (double)v.w);
        } else {
            za = make_double2((double)__uint_as_float(v.x), (double)__uint_as_float(v.y));
            zb = make_double2((double)__uint_as_float(v.z), (double)__uint_as_float(v.w));
        }
    } else {
        const unsigned char *p = plane_s + (size_t)idx * 32;
        za = load_sample<ENC>(p, 0, 0);
        zb = load_sample<ENC>(p, 1, 0);
    }
    if (pl.normalize) {
        za = normalize_sample(za, pl.norm_xmin, pl.norm_k);
        zb = normalize_sample(zb, pl.norm_xmin, pl.norm_k);
    }
}

// ------------------------------------------------------------------------------------ k_main
// grid.x = nchunks * ceil(ntiles / TPC); block = 32*W threads.  A CTA stages TPC consecutive
// tiles of one chunk in shared memory (raw bytes, once, shared by all rows); its warps then take
// (tile, row) items.  Lane roles follow the DMMA fragments: k = lane&3 owns the pairs
// [k*RL, (k+1)*RL) of block 8g + (lane>>2) in group g (B operand), and accumulates output row
// lane>>2 for blocks 8g + 2k, 8g + 2k + 1 (C operand).
template <int ENC, bool IQ>
__global__ void __launch_bounds__(256, 2)
k_main(const __grid_constant__ DevPlan pl, Scratch sc, const uint8_t *__restrict__ raw, int nchunks, int TPC)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, W = blockDim.x >> 5;
    const int q = pl.q, sb = pl.sb, RL = pl.RL;
    const int groups = (pl.ntiles + TPC - 1) / TPC;
    const int chunk = blockIdx.x / groups, tg = blockIdx.x % groups;
    if (chunk >= nchunks) return;
    const size_t tileb = main_tile_bytes(RL, sb), plane = main_plane_bytes(sb);
    unsigned char *warp_base = smem_raw + (size_t)TPC * tileb;
    const uint8_t *rawc = raw + (size_t)chunk * pl.N * sb;
    const int t0 = tg * TPC;
    const int ntl = min(TPC, pl.ntiles - t0);
    const int kq = lane & 3, nq = lane >> 2;
    // this lane's pair range inside a block: pairs [a0, a1), i.e. samples j and q-1-j
    const int a0 = min(kq * RL, pl.Hq), a1 = min((kq + 1) * RL, pl.Hq);
    const int npair = a1 - a0;                              // valid steps s < npair
    const int smid = (q & 1) && a1 == pl.Hq ? npair - 1 : -1;   // the step that holds the middle sample of an odd block

    // ---------------- stage the raw tiles (all warps, four rows in flight per lane), then (IQ) run
    //                  aggregates and block offsets
    if (sb == 2) stage_pairs<uint16_t>(smem_raw, tileb, rawc, t0, ntl, pl.ntiles, pl.cnt_last, q, pl.Hq, RL, pl.swap, warp, W, lane);
    else if (sb == 4) stage_pairs<uint32_t>(smem_raw, tileb, rawc, t0, ntl, pl.ntiles, pl.cnt_last, q, pl.Hq, RL, pl.swap, warp, W, lane);
    else if (sb == 8) stage_pairs<uint2>(smem_raw, tileb, rawc, t0, ntl, pl.ntiles, pl.cnt_last, q, pl.Hq, RL, pl.swap, warp, W, lane);
    else stage_pairs<uint4>(smem_raw, tileb, rawc, t0, ntl, pl.ntiles, pl.cnt_last, q, pl.Hq, RL, pl.swap, warp, W, lane);
    __syncthreads();
    for (int tl = warp; tl < ntl; tl += W) {
        const int t = t0 + tl;
        const int cnt = (t == pl.ntiles - 1) ? pl.cnt_last : SDRB_TB;
        unsigned char *tb = smem_raw + (size_t)tl * tileb;
        double2 *cl = reinterpret_cast<double2 *>(tb + (size_t)RL * plane);
        double2 *blkagg = cl + SDRB_TB;
        double2 excl = make_double2(0.0, 0.0);
        if (IQ) {
            // IQ-EMA aggregate of every block (the samples themselves stay uncorrected: the
            // corrector enters through the decoupled terms, DESIGN.md 3.3)
            for (int g = 0; g < 4; g++) {
                const int b = 8 * g + nq;
                double2 agg_a = make_double2(0.0, 0.0), agg_d = make_double2(0.0, 0.0);
                // ascending run = the first samples of the pairs (Horner); descending run = their
                // mirrors q-1-j, newest last: sum_sp lam^sp zb_sp (one decode pass for both)
                double wd = 1.0;
                for (int sp = 0; sp < npair; sp++) {
                    double2 za, zb;
                    load_pair<ENC>(pl, tb + (size_t)sp * plane, g, lane, za, zb);
                    agg_a.x = fma(pl.lam, agg_a.x, za.x); agg_a.y = fma(pl.lam, agg_a.y, za.y);
                    if (sp != smid) { agg_d.x = fma(wd, zb.x, agg_d.x); agg_d.y = fma(wd, zb.y, agg_d.y); }
                    wd *= pl.lam;
                }
                // EMA state at the 9 run boundaries of this block (all four lanes of the block
                // compute the same chain from the gathered run aggregates)
                const int base = lane & ~3;
                double2 A[9];
                A[0] = make_double2(0.0, 0.0);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const double2 v = shfl_c(agg_a, base + i);
                    A[i + 1] = make_double2(fma(pl.lam_run[i], A[i].x, v.x), fma(pl.lam_run[i], A[i].y, v.y));
                }
#pragma unroll
                for (int i = 4; i < 8; i++) {
                    const double2 v = shfl_c(agg_d, base + (7 - i));
                    A[i + 1] = make_double2(fma(pl.lam_run[i], A[i].x, v.x), fma(pl.lam_run[i], A[i].y, v.y));
                }
                if (kq == 0) blkagg[b] = A[8];
            }
            __syncwarp();
            const bool active = lane < cnt;
            double2 inc = active ? cscale(pl.Liq, blkagg[lane]) : make_double2(0.0, 0.0);
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const double2 tt = shfl_up_c(inc, 1 << i);
                if (lane >= (1 << i)) { inc.x = fma(pl.lamq_pow[i], tt.x, inc.x); inc.y = fma(pl.lamq_pow[i], tt.y, inc.y); }
            }
            excl = shfl_up_c(inc, 1);
            if (lane == 0) excl = make_double2(0.0, 0.0);
            const double2 tagg = shfl_c(inc, cnt - 1);
            if (lane == 0) sc.tile_agg[(size_t)chunk * pl.ntiles + t] = tagg;
        }
        cl[lane] = excl;
    }
    __syncthreads();

    // ---------------- items: (tile, row)
    double *xb = reinterpret_cast<double *>(warp_base + (size_t)warp * main_warp_bytes());
    double2 *x0s = reinterpret_cast<double2 *>(xb + 32 * SDRB_XSTRIDE);
    const int e = (lane >> 2) & 1, m = lane >> 3;
    for (int item = warp; item < ntl * pl.R; item += W) {
        const int tl = item % ntl, r = item / ntl;
        const int t = t0 + tl;
        const int cnt = (t == pl.ntiles - 1) ? pl.cnt_last : SDRB_TB;
        const unsigned char *tb = smem_raw + (size_t)tl * tileb;
        const double2 *cl = reinterpret_cast<const double2 *>(tb + (size_t)RL * plane);
        const double2 *T2r = pl.T2 + (size_t)r * q;
        const bool nco = pl.use_nco[r] != 0;

        // step s outside, the four block groups inside: the NCO phasors of the pair and the modal
        // A fragments are fetched once per step and serve 4 x 4 DMMAs
        double acc[4][8];
#pragma unroll
        for (int g = 0; g < 4; g++)
#pragma unroll
            for (int i = 0; i < 8; i++) acc[g][i] = 0.0;
        for (int sp = 0; sp < RL; sp++) {
            // steps past this lane's pairs (and the odd part of a middle sample) carry zero modal
            // coefficients and zero data: no selects in the loop
            const int j = a0 + sp;
            double2 Ta = make_double2(1.0, 0.0), Tb = Ta;
            if (nco && sp < npair) { Ta = __ldg(T2r + j); Tb = __ldg(T2r + (q - 1 - j)); }
            const double aE = __ldg(pl.Afrag + (size_t)(2 * sp) * 32 + lane);
            const double aO = __ldg(pl.Afrag + (size_t)(2 * sp + 1) * 32 + lane);
            const unsigned char *ps = tb + (size_t)sp * plane;
            const bool killb = pl.normalize && sp == smid;         // (a normalised zero is not zero)
            const bool first = sp == 0 && kq == 0;
#pragma unroll
            for (int g = 0; g < 4; g++) {
                double2 za, zb;
                load_pair<ENC>(pl, ps, g, lane, za, zb);
                if (first) x0s[8 * g + nq] = za;                   // first (raw) sample of the block
                if (killb) zb = make_double2(0.0, 0.0);
                const double2 ua = nco ? cmul(Ta, za) : za, ub = nco ? cmul(Tb, zb) : zb;
                const double2 a = cadd(ua, ub), d = csub(ua, ub);
                dmma884(acc[g][0], acc[g][1], aE, a.x);
                dmma884(acc[g][2], acc[g][3], aE, a.y);
                dmma884(acc[g][4], acc[g][5], aO, d.x);
                dmma884(acc[g][6], acc[g][7], aO, d.y);
            }
        }
        // combine the four real sums into F/G (part e of poles m and m+4), exchange
#pragma unroll
        for (int g = 0; g < 4; g++) {
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const int b = 8 * g + 2 * kq + i;
                const double Sr = acc[g][i], Si = acc[g][2 + i], Dr = acc[g][4 + i], Di = acc[g][6 + i];
                const double oS = __shfl_xor_sync(0xffffffffu, Si, 4);
                const double oD = __shfl_xor_sync(0xffffffffu, Di, 4);
                double Sup, Slo, Dup, Dlo;
                if (e == 0) { Sup = Sr - oS; Slo = Sr + oS; Dup = Dr - oD; Dlo = Dr + oD; }
                else        { Sup = oS + Sr; Slo = oS - Sr; Dup = oD + Dr; Dlo = oD - Dr; }
                const double Fu = Sup + Dup, Gu = Sup - Dup, Fl = Slo + Dlo, Gl = Slo - Dlo;
                xb[(2 * m + e) * SDRB_XSTRIDE + b] = Fu;
                xb[(2 * (m + 4) + e) * SDRB_XSTRIDE + b] = Fl;
                xb[(2 * (8 + m) + e) * SDRB_XSTRIDE + b] = Gu;
                xb[(2 * (12 + m) + e) * SDRB_XSTRIDE + b] = Gl;
            }
        }
        __syncwarp();
        // tile-local scans in the rotating frame: lanes 0..7 forward poles, 8..15 backward
        if (lane < 16) {
            const bool fwd = lane < 8;
            const double2 Pm = pl.Prot[(size_t)r * 16 + lane];
            double2 st = make_double2(0.0, 0.0);
            // forward lanes: exclusive scan = the inclusive one stored one slot up (slot 0 = 0, slot
            // cnt is padding or an unused block); backward lanes: inclusive, in place.  The next
            // input is fetched before the store that may overwrite it.
            const int dir = fwd ? 1 : -1;
            double *xr = xb + (2 * lane) * SDRB_XSTRIDE + (fwd ? 0 : cnt - 1), *xi = xr + SDRB_XSTRIDE;
            double *orr = xr + (fwd ? 1 : 0), *oi = orr + SDRB_XSTRIDE;
            double2 v = make_double2(*xr, *xi);
            if (fwd) { *xr = 0.0; *xi = 0.0; }
            for (int step = 0; step < cnt; step++) {
                xr += dir; xi += dir;
                double2 vn = make_double2(0.0, 0.0);
                if (step + 1 < cnt) vn = make_double2(*xr, *xi);
                st = cfma(Pm, st, v);
                *orr = st.x; *oi = st.y;
                orr += dir; oi += dir;
                v = vn;
            }
            if (fwd) st = cmul(pl.T3[(size_t)r * (SDRB_TB + 1) + cnt - 1], st);
            sc.agg[(((size_t)chunk * pl.R + r) * pl.ntiles + t) * 16 + lane] = st;
        }
        __syncwarp();
        // partial outputs, lane <-> block
        if (lane < cnt) {
            double2 sw = make_double2(0.0, 0.0), sT = make_double2(0.0, 0.0);
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const double2 Wv = make_double2(xb[(2 * i) * SDRB_XSTRIDE + lane], xb[(2 * i + 1) * SDRB_XSTRIDE + lane]);
                const double2 Tv = make_double2(xb[(2 * (8 + i)) * SDRB_XSTRIDE + lane], xb[(2 * (8 + i) + 1) * SDRB_XSTRIDE + lane]);
                sw = cfma(pl.rb[(size_t)r * 8 + i], Wv, sw);
                sT = cfma(pl.rbT[(size_t)r * 8 + i], Tv, sT);
            }
            const double2 epsb = cconj(pl.T3[(size_t)r * (SDRB_TB + 1) + 1]);
            const double2 x0 = x0s[lane];
            double2 ys = cfma(epsb, sw, sT);
            ys.x = fma(pl.g0, x0.x, ys.x); ys.y = fma(pl.g0, x0.y, ys.y);
            if (IQ) {                                  // - gamma * (tile-local offset at this block)
                const double2 gm = pl.gamma[r], o = cl[lane];
                ys = cfma(make_double2(-gm.x, -gm.y), o, ys);
            }
            const double2 yp = cmul(pl.T3[(size_t)r * (SDRB_TB + 1) + lane], ys);
            sc.ypart[((size_t)chunk * pl.R + r) * pl.Mf + (size_t)t * SDRB_TB + lane] = yp;
        }
        __syncwarp();
    }
}

// -------------------------------------------------------------------------------- IQ kernels
// The offsets over one chunk's tiles, warp <-> chunk: lane <-> run [t0, t1) of per = ceil(nt/32)
// consecutive tiles (per = 1 whenever nt <= 32), whose maps o -> lam_tile o + agg[t] the lane folds
// serially before the warp composes the runs.  From o0, the offset at the chunk start: `in` = the
// offset entering tile t0, `end` = the offset at q*Mf; `gain` = the composed offset term of the whole
// chunk (the offset it gains from a zero start).
struct TileOffsets {
    double2 in, end, gain;
    int t0, t1;
};
__device__ __forceinline__ TileOffsets tile_offsets(const DevPlan &pl, const double2 *ta, double2 o0, int lane)
{
    const int nt = pl.ntiles, per = (nt + 31) >> 5;
    TileOffsets r;
    r.t0 = min(nt, lane * per);
    r.t1 = min(nt, r.t0 + per);
    double m = 1.0;
    double2 a = make_double2(0.0, 0.0);
    if (r.t0 < r.t1) { m = pl.lam_tile[r.t0 == nt - 1 ? 1 : 0]; a = ta[r.t0]; }
#pragma unroll 4         // (a deeper unroll costs k_iqgain its 32-register budget)
    for (int t = r.t0 + 1; t < r.t1; t++) {
        const double lt = pl.lam_tile[t == nt - 1 ? 1 : 0];
        const double2 g = ta[t];
        a.x = fma(lt, a.x, g.x); a.y = fma(lt, a.y, g.y);
        m *= lt;
    }
    warp_affine_scan(m, a, lane);
    const int last = 31 - __clz(__ballot_sync(0xffffffffu, r.t0 < r.t1));   // the lane with tile nt-1
    const double2 incl = make_double2(fma(m, o0.x, a.x), fma(m, o0.y, a.y));   // offset leaving tile t1-1
    r.in = shfl_up_c(incl, 1);
    if (lane == 0) r.in = o0;
    r.end = shfl_c(incl, last);
    r.gain = shfl_c(a, last);
    return r;
}

// k_iqgain: warp <-> chunk, the offset gained over the chunk from a zero state -> gain[c]: the tile
// maps, then the samples of the partial block (one lane, serially).  At most 32 registers: 8 CTAs
// per SM, so that a batch of 8192 chunks runs in one wave.
template <int ENC>
__global__ void __launch_bounds__(256, 8)
k_iqgain(const __grid_constant__ DevPlan pl, Scratch sc, const uint8_t *__restrict__ raw, int nchunks)
{
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= nchunks) return;
    double2 o = tile_offsets(pl, sc.tile_agg + (size_t)c * pl.ntiles, make_double2(0.0, 0.0), lane).gain;
    if (lane != 0) return;
    if (pl.rem) {
        const uint8_t *rawc = raw + (size_t)c * pl.N * pl.sb;
        double2 acc = make_double2(0.0, 0.0);
        for (int j = 0; j < pl.rem; j++) {
            const double2 z = decode_sample<ENC>(pl, rawc, (long)pl.q * pl.Mf + j);
            acc.x = fma(pl.lam, acc.x, z.x); acc.y = fma(pl.lam, acc.y, z.y);
        }
        const double lr = pl.lam_j[pl.rem];
        o.x = fma(lr, o.x, pl.Liq * acc.x); o.y = fma(lr, o.y, pl.Liq * acc.y);
    }
    sc.gain[c] = o;
}

// k_iqchunk: warp <-> chunk: the offset a whole chunk gains from a zero state, straight from the raw
// bytes (decode, normalise, EMA) -> gain[c].  The pre-pass of time-segment sharding for streams
// longer than one batch (sdrb_iq_gain): no outputs, the raw bytes are read once.
template <int ENC>
__global__ void __launch_bounds__(256)
k_iqchunk(const __grid_constant__ DevPlan pl, Scratch sc, const uint8_t *__restrict__ raw, int nchunks)
{
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= nchunks) return;
    const uint8_t *rawc = raw + (size_t)c * pl.N * pl.sb;
    // lane <-> contiguous run of ceil(N/32) samples
    const int per = (pl.N + 31) / 32;
    const int n0 = min(pl.N, lane * per), n1 = min(pl.N, n0 + per);
    double2 a = make_double2(0.0, 0.0);
    double m = 1.0;
    for (int n = n0; n < n1; n++) {
        const double2 z = decode_sample<ENC>(pl, rawc, n);
        a.x = fma(pl.lam, a.x, z.x); a.y = fma(pl.lam, a.y, z.y);
        m *= pl.lam;
    }
    warp_affine_scan(m, a, lane);
    if (lane == 31) sc.gain[c] = make_double2(pl.Liq * a.x, pl.Liq * a.y);
}

// k_iqscan_c: one CTA of 1024 threads; exclusive scan of the per-chunk maps o -> lam_N o + gain[c]
// from the handle's IQ state -> start[c] and the new state.  8 chunks per thread and round (their
// gains are loaded together).
__global__ void __launch_bounds__(1024)
k_iqscan_c(const __grid_constant__ DevPlan pl, Scratch sc, int nchunks)
{
    __shared__ double2 s_a[32];
    __shared__ double s_m[32];
    __shared__ double2 s_state;
    const int tid = threadIdx.x;
    const double2 *__restrict__ gain = sc.gain;
    double2 *__restrict__ start = sc.start;
    if (tid == 0) s_state = sc.iq_state[0];
    __syncthreads();
    for (int base = 0; base < nchunks; base += 1024 * 8) {
        const int c0 = base + tid * 8;
        double2 g[8];
#pragma unroll
        for (int i = 0; i < 8; i++) g[i] = (c0 + i < nchunks) ? gain[c0 + i] : make_double2(0.0, 0.0);
        double m = 1.0;
        double2 a = make_double2(0.0, 0.0);
#pragma unroll
        for (int i = 0; i < 8; i++)
            if (c0 + i < nchunks) { a.x = fma(pl.lam_N, a.x, g[i].x); a.y = fma(pl.lam_N, a.y, g[i].y); m *= pl.lam_N; }
        double em, tm;
        double2 ea, ta;
        block_affine_scan(m, a, s_m, s_a, em, ea, tm, ta);
        const double2 st0 = s_state;
        double2 o = make_double2(fma(em, st0.x, ea.x), fma(em, st0.y, ea.y));
#pragma unroll
        for (int i = 0; i < 8; i++)
            if (c0 + i < nchunks) {
                start[c0 + i] = o;
                o.x = fma(pl.lam_N, o.x, g[i].x); o.y = fma(pl.lam_N, o.y, g[i].y);
            }
        __syncthreads();
        if (tid == 1023) s_state = make_double2(fma(tm, st0.x, ta.x), fma(tm, st0.y, ta.y));
        __syncthreads();
    }
    if (tid == 0) sc.iq_state[0] = s_state;
}

// k_iqtiles: warp <-> chunk, offsets at the tile starts from the chunk-start offset start[c].
__global__ void __launch_bounds__(256)
k_iqtiles(const __grid_constant__ DevPlan pl, Scratch sc, int nchunks)
{
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= nchunks) return;
    const int nt = pl.ntiles;
    const double2 *ta = sc.tile_agg + (size_t)c * nt;
    double2 *ot = sc.off_tile + (size_t)c * (nt + 1);
    const TileOffsets to = tile_offsets(pl, ta, sc.start[c], lane);
    double2 o = to.in;
    for (int t = to.t0; t < to.t1; t++) {
        ot[t] = o;
        const double lt = pl.lam_tile[t == nt - 1 ? 1 : 0];
        const double2 g = ta[t];
        o.x = fma(lt, o.x, g.x); o.y = fma(lt, o.y, g.y);
    }
    if (to.t0 < to.t1 && to.t1 == nt) ot[nt] = to.end;      // offset at sample q*Mf
}

// Time-segment sharding (SURVEY 8e): the IQ offset a segment gained from a zero start, and the
// fold of the gains of the segments before this rank's into its start offset -- on the device, so
// that the exchange between the two passes needs no host round trip.
__global__ void k_iq_export(Scratch sc, double *dst3, double nsamples)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const double2 g = sc.iq_state[0];
        dst3[0] = g.x; dst3[1] = g.y; dst3[2] = nsamples;
    }
}
__global__ void k_iq_prefix(Scratch sc, const double *gains3, int rank, double lam)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double2 off = make_double2(0.0, 0.0);
        for (int i = 0; i < rank; i++) {
            const double d = pow(lam, gains3[3 * i + 2]);
            off.x = fma(d, off.x, gains3[3 * i]); off.y = fma(d, off.y, gains3[3 * i + 1]);
        }
        sc.iq_state[0] = off;
    }
}

// ------------------------------------------------------------------------- chunk boundary
// sosfiltfilt's boundary at a chunk's two edges, written once for k_finish, k_fixup and the seamless
// kernels: lane <-> sample for the edge samples, lane = (mode, quarter of the terms) for the closed
// forms of the boundary recurrences.  The front ends sum the UNcorrected rotated samples, so their
// frame has W~ = (w + alpha s) / beta and T~ = (T + alphaT s) / betaT, s = off[n] e^{jwn} (DESIGN.md
// 3.3); the callers convert.

struct EdgeSample {
    double2 x;      // this lane's sample, IQ-corrected and rotated
    double2 o;      // the offset after the window when it ends running forward: the next round's o
};

// A window of n <= 32 samples, lane <-> sample; z = this lane's decoded sample (zero past the
// window).  read_file.py:72-77 is the linear recurrence off' = lam off + L z; from o, the offset at
// sample n_bwd, lanes below n_bwd run it BACKWARD, off_m = mu^(n_bwd-m) o - L mu sum_{m<=i<n_bwd}
// mu^(i-m) z_i (mu = 1/lam), lanes from n_bwd on forward, off_m = lam^(m-n_bwd) o + L
// sum_{n_bwd<=i<m} lam^(m-1-i) z_i: a 5-level warp scan for each direction the window has.  The
// corrected sample is then rotated by E, this lane's NCO phase.
__device__ __forceinline__ EdgeSample edge_correct(const DevPlan &pl, double2 z, double2 o, int n, int n_bwd, double2 E,
                                                   int lane)
{
    EdgeSample e{z, o};
    if (pl.correct_iq) {
        const double2 zero = make_double2(0.0, 0.0);
        if (n_bwd > 0) {
            double2 B = lane < n_bwd ? z : zero;
#pragma unroll
            for (int lv = 0; lv < 5; lv++) {
                const double2 td = make_double2(__shfl_down_sync(0xffffffffu, B.x, 1 << lv), __shfl_down_sync(0xffffffffu, B.y, 1 << lv));
                if (lane + (1 << lv) < 32) { B.x = fma(pl.mu_pw[1 << lv], td.x, B.x); B.y = fma(pl.mu_pw[1 << lv], td.y, B.y); }
            }
            if (lane < n_bwd) {
                const double mun = pl.mu_pw[n_bwd - lane], lm = pl.Liq * pl.mu_pw[1];
                e.x.x -= fma(mun, o.x, -lm * B.x); e.x.y -= fma(mun, o.y, -lm * B.y);
            }
        }
        if (n_bwd < n) {
            double2 S = lane >= n_bwd ? z : zero;
#pragma unroll
            for (int lv = 0; lv < 5; lv++) {
                const double2 tu = shfl_up_c(S, 1 << lv);
                if (lane >= (1 << lv)) { S.x = fma(pl.lam_pw[1 << lv], tu.x, S.x); S.y = fma(pl.lam_pw[1 << lv], tu.y, S.y); }
            }
            double2 Sx = shfl_up_c(S, 1);
            if (lane == 0) Sx = zero;
            if (lane >= n_bwd) {
                const double lamn = pl.lam_pw[lane - n_bwd];
                e.x.x -= fma(lamn, o.x, pl.Liq * Sx.x); e.x.y -= fma(lamn, o.y, pl.Liq * Sx.y);
            }
            const double2 Sn = shfl_c(S, n - 1);
            const double ln = pl.lam_pw[n - n_bwd];
            e.o = make_double2(fma(ln, o.x, pl.Liq * Sn.x), fma(ln, o.y, pl.Liq * Sn.y));
        }
    }
    if (lane < n) e.x = cmul(e.x, E);
    return e;
}

struct BoundarySums {
    double2 A, B, C;
};

// The closed forms of the serial boundary recurrences against pk[k][i] = p_i^k, lane = (mode i =
// lane & 7, quarter lane >> 3 of the terms); every lane returns its mode's sums.  Head, from its odd
// extension ha[0..nh): A = w(edge) = p^nh zhat ha[0] + sum_j p^(nh-1-j) ha[j].  End, from the sequence
// seq[0..nseq) (the partial block, then the tail extension): B = T at q*Mf = sum_k p^k seq[k], and
// C = sum_{k <= nseq-2} p^(nseq-2-k) seq[k], the sequence's part of w(L-2).  nh = 0 or nseq = 0
// skips that end.
__device__ __forceinline__ BoundarySums boundary_sums(const DevPlan &pl, const double2 *pk, const double2 *ha, int nh,
                                                      const double2 *seq, int nseq, int lane)
{
    const int i8 = lane & 7, sub = lane >> 3;
    const int dh = (nh + 3) >> 2, ds = (nseq + 3) >> 2;     // terms per quarter
    const int h0 = sub * dh, h1 = min(nh, h0 + dh), s0 = sub * ds, s1 = min(nseq, s0 + ds);
    BoundarySums s;
    s.A = s.B = s.C = make_double2(0.0, 0.0);
    for (int u = 0; u < max(dh, ds); u++) {
        const int j = h0 + u, k = s0 + u;
        if (j < h1) s.A = cfma(pk[(nh - 1 - j) * 8 + i8], ha[j], s.A);
        if (k < s1) {
            const double2 b = seq[k];
            s.B = cfma(pk[k * 8 + i8], b, s.B);
            if (k <= nseq - 2) s.C = cfma(pk[(nseq - 2 - k) * 8 + i8], b, s.C);
        }
    }
#pragma unroll
    for (int sft = 8; sft < 32; sft <<= 1) {
        s.A = cadd(s.A, shfl_xor_c(s.A, sft));
        s.B = cadd(s.B, shfl_xor_c(s.B, sft));
        s.C = cadd(s.C, shfl_xor_c(s.C, sft));
    }
    if (nh > 0) s.A = cfma(pk[nh * 8 + i8], cmul(pl.zhat[i8], ha[0]), s.A);
    return s;
}

// sosfiltfilt's boundary vector zeta_i (mode i = lane & 7) from W, the true forward state of mode i at
// q*Mf, and C of boundary_sums over seq[0..nseq): w(L-2) = p^(nseq-1) W + C, w(L-1) one step on, and
// zeta = zhat y_f(L-1) - xi w(L-1), y_f(L-1) = sum_l c_l w_l(L-2) + d seq[nseq-1].  The modes' values
// are those of lanes 0..7; all 32 lanes must call it.
__device__ __forceinline__ double2 boundary_zeta(const DevPlan &pl, const double2 *pk, const double2 *seq, int nseq,
                                                 double2 W, double2 C, int lane)
{
    const int i8 = lane & 7;
    const double2 last = seq[nseq - 1];
    const double2 wL1 = cfma(pk[(nseq - 1) * 8 + i8], W, C);
    const double2 wL = cfma(pl.p[i8], wL1, last);
    double2 part = cmul(pl.c[i8], wL1);
    for (int sft = 1; sft < 8; sft <<= 1) part = cadd(part, shfl_xor_c(part, sft));
    const double2 yfL1 = make_double2(fma(pl.d, last.x, part.x), fma(pl.d, last.y, part.y));
    double2 za = cmul(pl.zhat[i8], yfL1), zb = make_double2(0.0, 0.0);
#pragma unroll
    for (int l = 0; l < 8; l += 2) {
        za = csub(za, cmul(pl.xi[i8 * 8 + l], shfl_c(wL, l)));
        zb = csub(zb, cmul(pl.xi[i8 * 8 + l + 1], shfl_c(wL, l + 1)));
    }
    return cadd(za, zb);
}

// The general kernels' head: z = lane n's decoded sample n <= edge, o = the offset at sample 0; the
// odd extension 2 x[0] - x[edge-j], j < edge, of the corrected rotated samples -> ha.
__device__ __forceinline__ void head_window(const DevPlan &pl, int r, double2 z, double2 o, double2 *ha, int lane)
{
    const int edge = pl.edge;
    const double2 E = lane <= edge ? pl.Ehead[(size_t)r * (edge + 1) + lane] : make_double2(0.0, 0.0);
    const double2 x = edge_correct(pl, z, o, edge + 1, 0, E, lane).x;
    const double2 x0 = shfl_c(x, 0), xa = shfl_c(x, max(0, edge - lane));
    if (lane < edge) ha[lane] = make_double2(fma(2.0, x0.x, -xa.x), fma(2.0, x0.y, -xa.y));
    __syncwarp();
}

// The general kernels' end window: samples ws..N-1 -> s[0..nend), corrected from o, the offset at
// q*Mf (backward below nend - rem, forward from there), in rounds of 32 that carry the offset, then
// the tail extension 2 x[N-1] - x[N-2-j], j < edge -> s[nend..nend+edge).  load(j) decodes window
// sample j.  The end sequence of boundary_sums is s + nend - rem, rem + edge samples long.
template <class Load>
__device__ __forceinline__ void end_window(const DevPlan &pl, int r, Load load, double2 o, double2 *s, int lane)
{
    const int nend = pl.nend;
    // a window longer than one round has rem = nend: forward throughout
    for (int j0 = 0; j0 < nend; j0 += 32) {
        const int j = j0 + lane;
        double2 z = make_double2(0.0, 0.0), E = z;
        if (j < nend) { z = load(j); E = pl.Eend[(size_t)r * nend + j]; }
        const EdgeSample e = edge_correct(pl, z, o, min(32, nend - j0), nend - pl.rem, E, lane);
        if (j < nend) s[j] = e.x;
        o = e.o;
    }
    __syncwarp();
    const double2 xN1 = s[nend - 1];
    for (int k = lane; k < pl.edge; k += 32) {
        const double2 b = s[nend - 2 - k];
        s[nend + k] = make_double2(fma(2.0, xN1.x, -b.x), fma(2.0, xN1.y, -b.y));
    }
    __syncwarp();
}

// Mode i's carries across a chunk's tiles from the state w at one end: forward from tile 0 (the
// carry-in of tile t goes to slot t, column i) or backward from q*Mf (slot t+1, column 8+i; the state
// at tile 0 to slot 0).  store(slot * 16 + column, be w) keeps them, pre-scaled by beta / betaT for
// the outputs; returns the state at the other end.
template <class Store>
__device__ __forceinline__ double2 tile_carries(const DevPlan &pl, const double2 *T1, const double2 *agg, int i,
                                                bool fwd, double2 be, double2 w, Store store)
{
    const int nt = pl.ntiles, o = fwd ? i : 8 + i;
    for (int s = 0; s < nt; s++) {
        const int t = fwd ? s : nt - 1 - s;
        store((size_t)(fwd ? t : t + 1) * 16 + o, cmul(be, w));
        const int cnt = (t == nt - 1) ? pl.cnt_last : SDRB_TB;
        w = cfma(pl.Ppow[(size_t)cnt * 8 + i], w, cmul(T1[t], agg[(size_t)t * 16 + o]));
    }
    if (!fwd) store((size_t)o, cmul(be, w));
    return w;
}

// Outputs at the full-block starts k = first, first + stride, .. < Mf (tile t, block l):
// T1 (ypart - off psiY) + sum RW Win + RT Tn, plus bnd zeta from k = k_bnd on; each goes to store(k, v).
template <class Store>
__device__ __forceinline__ void block_outputs(const DevPlan &pl, int r, const double2 *ypart, const double2 *offt,
                                              const double2 *T1, const double2 *carry, const double2 *zeta,
                                              int k_bnd, int first, int stride, Store store)
{
    const int nt = pl.ntiles;
    for (int k = first; k < pl.Mf; k += stride) {
        const int t = k / SDRB_TB, l = k % SDRB_TB;
        const int kind = (t == nt - 1) ? 1 : 0;
        const int cnt = kind ? pl.cnt_last : SDRB_TB;
        double2 v = ypart[k];
        if (pl.correct_iq) {
            const double2 s = make_double2(-offt[t].x, -offt[t].y);
            v = cfma(s, pl.psiY[((size_t)kind * pl.R + r) * SDRB_TB + l], v);
        }
        v = cmul(T1[t], v);
        const double2 *Win = carry + (size_t)t * 16, *Tn = carry + (size_t)(t + 1) * 16 + 8;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            v = cfma(pl.RW[(size_t)l * 8 + i], Win[i], v);
            v = cfma(pl.RT[(size_t)(cnt - l) * 8 + i], Tn[i], v);
        }
        if (k >= k_bnd) {
#pragma unroll
            for (int i = 0; i < 8; i++) v = cfma(pl.bnd[(size_t)k * 8 + i], zeta[i], v);
        }
        store(k, v);
    }
}

// ----------------------------------------------------------------------------------- k_fixup
// One CTA per (chunk, row).  Warp 0 runs the chunk boundary: the head and the end window lane <->
// sample, the boundary sums; lanes 0..7 <-> modes run the forward carries, zeta, the partial block's
// output and the backward carries; then all threads emit the outputs at the full-block starts.
template <int ENC>
__global__ void __launch_bounds__(128)
k_fixup(const __grid_constant__ DevPlan pl, Scratch sc, const uint8_t *__restrict__ raw, int nchunks)
{
    __shared__ double2 s_x[SDRB_NEDGE];    // head extension (edge), then end window (nend) + tail extension (edge)
    __shared__ double2 s_zeta[SDRB_NP];
    const int chunk = blockIdx.x / pl.R, r = blockIdx.x % pl.R;
    if (chunk >= nchunks) return;
    const int nt = pl.ntiles, edge = pl.edge;
    const uint8_t *rawc = raw + (size_t)chunk * pl.N * pl.sb;
    const double2 *offt = sc.off_tile + (size_t)chunk * (nt + 1);
    const double2 *aggr = sc.agg + ((size_t)chunk * pl.R + r) * nt * 16;
    double2 *carry = sc.carry + ((size_t)chunk * pl.R + r) * (nt + 1) * 16;
    double2 *yrow = sc.y + ((size_t)chunk * pl.R + r) * pl.M;
    const double2 *T1r = pl.T1 + (size_t)r * nt;
    double2 *s_ha = s_x, *s_e = s_x + edge;

    if (threadIdx.x < 32) {
        const int lane = threadIdx.x, i = lane & 7;
        const bool iq = pl.correct_iq != 0;
        const double2 o0 = offt[0], oE = offt[nt];
        head_window(pl, r, lane <= edge ? decode_sample<ENC>(pl, rawc, lane) : make_double2(0.0, 0.0), o0, s_ha, lane);
        end_window(pl, r, [&](int j) { return decode_sample<ENC>(pl, rawc, (long)pl.ws + j); }, oE, s_e, lane);
        const double2 *seq = s_e + pl.nend - pl.rem;
        const int nseq = pl.rem + edge;
        const BoundarySums bs = boundary_sums(pl, pl.pk, s_ha, edge, seq, nseq, lane);
        double2 w = iq ? cmul(cfma(pl.alpha[(size_t)r * 8 + i], o0, bs.A), pl.binv[(size_t)r * 8 + i]) : bs.A;
        auto keep = [&](size_t j, double2 v) { carry[j] = v; };
        if (lane < 8) w = tile_carries(pl, T1r, aggr, i, true, pl.beta[(size_t)r * 8 + i], w, keep);
        // at q*Mf: the true forward state, and the anticausal state into the T~ frame
        const double2 sE = iq ? cmul(oE, pl.phE[r]) : make_double2(0.0, 0.0);
        if (iq) w = csub(cmul(pl.beta[(size_t)r * 8 + i], w), cmul(pl.alpha[(size_t)r * 8 + i], sE));
        const double2 Tt = iq ? cmul(cfma(pl.alphaT[(size_t)r * 8 + i], sE, bs.B), pl.binvT[(size_t)r * 8 + i]) : bs.B;
        const double2 zeta = boundary_zeta(pl, pl.pk, seq, nseq, w, bs.C, lane);
        if (lane < 8) s_zeta[i] = zeta;
        if (pl.rem) {       // the output at the partial block
            double2 v = cfma(pl.rho[i], w, cmul(pl.rho_p[i], bs.B));
            v = cfma(pl.bnd[(size_t)pl.Mf * 8 + i], zeta, v);
            for (int sft = 1; sft < 8; sft <<= 1) v = cadd(v, shfl_xor_c(v, sft));
            if (lane == 0) yrow[pl.Mf] = make_double2(fma(pl.g0, seq[0].x, v.x), fma(pl.g0, seq[0].y, v.y));
        }
        if (lane < 8) tile_carries(pl, T1r, aggr, i, false, pl.betaT[(size_t)r * 8 + i], Tt, keep);
    }
    __syncthreads();
    block_outputs(pl, r, sc.ypart + ((size_t)chunk * pl.R + r) * pl.Mf, offt, T1r, carry, s_zeta, pl.k_bnd,
                  threadIdx.x, blockDim.x, [&](int k, double2 v) { yrow[k] = v; });
}

// ----------------------------------------------------------------------------------- k_demod
// k_demod's row scratch (bytes), in shared memory or, when it does not fit, per CTA in global
// memory: the output row of M doubles, then two FFT buffers of ceil(M/4) complex points (fm: the
// first holds the M/2 pair phases as doubles).
__host__ __device__ inline size_t demod_smem_bytes(int M) { return (size_t)4 * ((M + 3) / 4) * sizeof(double2); }

// One CTA per (chunk, row): y[M] complex -> out[row][chunk*M .. +M) doubles.
// Generic entry used both by the chain (y from sc.y) and by the module-level operators.  The iq
// instance (OUT_IQ) frames y itself as out[row][chunk*2M .. +2M): (Re, Im) pairs, no output
// low-pass.  The output filter (up to 4 sections) runs on warp 0, lane <-> segment of Lseg outputs
// (sdrb_outstage.cuh); the usb / lsb instance (OUT_SSB) runs it as the complex band-pass on y itself.
template <int OUT>
__global__ void __launch_bounds__(256)
k_demod(const __grid_constant__ DevPlan pl, const double2 *__restrict__ yall, double *__restrict__ out,
        double2 *scratch, int nchunks, int demod, int apply_sos, int be_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int chunk = blockIdx.x / pl.R, r = blockIdx.x % pl.R;
    if (chunk >= nchunks) return;
    const int M = pl.M, h = M >> 1;
    const double2 *y = yall + ((size_t)chunk * pl.R + r) * M;
    if constexpr (OUT == OUT_IQ) {
        double2 *o2 = reinterpret_cast<double2 *>(out + ((size_t)r * nchunks + chunk) * 2 * M);
        for (int k = threadIdx.x; k < M; k += blockDim.x) frame_store(o2 + k, y[k], be_out);
        return;
    }
    const int nq = (M + 3) >> 2;
    double2 *row = pl.demod_in_smem ? reinterpret_cast<double2 *>(smem_raw) : scratch + (size_t)blockIdx.x * 4 * nq;
    double *z = reinterpret_cast<double *>(row);
    double2 *fa = row + 2 * nq, *fb = fa + nq;
    if (OUT == OUT_REAL && demod == 0) {   // fm: demodulation.py:25-38
        // the pair phases are also the even outputs of the FFT interpolation (the dense matrix
        // overwrites them)
        double *ph = reinterpret_cast<double *>(fa);
        for (int i = threadIdx.x; i < h; i += blockDim.x) {
            const double v = pair_phase(y[2 * i], y[2 * i + 1]);
            ph[i] = v;
            z[2 * i] = v;
        }
        __syncthreads();
        if (pl.fft_ok) {
            fm_interp2x(fa, fb, M, pl.tw, CtaGroup{(int)threadIdx.x, (int)blockDim.x},
                        [&](int k, double v) { z[k] = v; });
        } else {
            // dense interpolation matrix built by the host from scipy.signal.resample
            for (int k = threadIdx.x; k < M; k += blockDim.x) {
                const double *wrow = pl.fm_interp + (size_t)k * h;
                double acc = 0.0;
                for (int i = 0; i < h; i++) acc = fma(wrow[i], ph[i], acc);
                z[k] = acc;
            }
        }
    } else if (OUT == OUT_REAL) {          // am | re | im
        for (int k = threadIdx.x; k < M; k += blockDim.x) z[k] = demod_scalar(y[k], demod);
    }
    __syncthreads();
    if ((OUT == OUT_SSB || (apply_sos && pl.nsec_out > 0)) && threadIdx.x < 32) {
        const int lane = threadIdx.x, Ls = pl.sos_Lseg, lo = min(M, lane * Ls);
        std::conditional_t<OUT == OUT_SSB, double2, double> st[8];
        sos_segments(
            pl, pl.nsec_out, lo, min(M, lo + Ls) - lo, lane,
            [&](int j) {
                if constexpr (OUT == OUT_SSB) return y[lo + j];
                else return z[lo + j];
            },
            [&](int j) -> double & { return z[lo + j]; }, st);
    }
    __syncthreads();
    double *o = out + ((size_t)r * nchunks + chunk) * M;
    for (int k = threadIdx.x; k < M; k += blockDim.x) frame_store(o + k, z[k], be_out);
}

// demodulation.py:71-79  res[m,n] = y[n] * shift[m,n]
__global__ void k_shift(const double2 *__restrict__ y, const double2 *__restrict__ shift,
                        double2 *__restrict__ res, int R, int N)
{
    const size_t total = (size_t)R * N;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const double2 a = y[idx % N], b = shift[idx];
        res[idx] = make_double2(__dadd_rn(__dmul_rn(a.x, b.x), -__dmul_rn(a.y, b.y)),
                                __dadd_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x)));
    }
}

// read_file.py:100-101  z = y['re'] + 1j*y['im'] on the structured view of the raw bytes.
template <int ENC>
__global__ void k_decode(const uint8_t *__restrict__ raw, double2 *__restrict__ z, size_t n, int swap)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        z[i] = load_sample<ENC>(raw, (long)i, swap);
}

// read_file.py:65-77 / extra/src/iq_correction.pyx:46-52: z[i] -= off; off += z[i] * L, as the
// linear recurrence off' = lam off + L z evaluated by one CTA: thread <-> contiguous run, affine
// maps scanned across the threads, second pass applies the offsets.
__global__ void __launch_bounds__(1024)
k_correct_iq(double2 *__restrict__ z, size_t n, double2 *__restrict__ off_io, double L)
{
    __shared__ double2 s_a[32];
    __shared__ double s_m[32];
    const int tid = threadIdx.x;
    const double lam = 1.0 - L;
    const size_t per = (n + blockDim.x - 1) / blockDim.x;
    const size_t i0 = min(n, (size_t)tid * per), i1 = min(n, i0 + per);
    double2 a = make_double2(0.0, 0.0);
    double m = 1.0;
    for (size_t i = i0; i < i1; i++) {
        const double2 v = z[i];
        a.x = fma(lam, a.x, L * v.x); a.y = fma(lam, a.y, L * v.y);
        m *= lam;
    }
    double em, tm;
    double2 ea, ta;
    block_affine_scan(m, a, s_m, s_a, em, ea, tm, ta);
    const double2 st0 = off_io[0];
    double2 o = make_double2(fma(em, st0.x, ea.x), fma(em, st0.y, ea.y));
    for (size_t i = i0; i < i1; i++) {
        double2 v = z[i];
        v.x -= o.x; v.y -= o.y;
        o.x = fma(v.x, L, o.x); o.y = fma(v.y, L, o.y);
        z[i] = v;
    }
    __syncthreads();
    if (tid == blockDim.x - 1) off_io[0] = o;
}

// dsp_processor.py:159-160  z[:] = savgol_filter(z, window, 3) per chunk row of M outputs, as the
// three linear maps SciPy uses (tab = head rows | FIR row | tail rows, each `w` long).
__global__ void k_savgol(const double *__restrict__ x, double *__restrict__ y, const double *__restrict__ tab,
                         int w, int nhead, int ntail, int lo, int M, size_t nseg)
{
    for (size_t seg = blockIdx.x; seg < nseg; seg += gridDim.x) {
        const double *xs = x + seg * M;
        double *ys = y + seg * M;
        for (int k = threadIdx.x; k < M; k += blockDim.x) {
            int row, base;
            if (k < nhead) { row = k; base = 0; }
            else if (k >= M - ntail) { row = nhead + 1 + (k - (M - ntail)); base = M - w; }
            else { row = nhead; base = k + lo; }
            const double *sr = tab + (size_t)row * w;
            double acc = 0.0;
            for (int j = 0; j < w; j++) {
                const int i = base + j;
                if (i >= 0 && i < M) acc = fma(sr[j], xs[i], acc);
            }
            ys[k] = acc;
        }
    }
}
