// sdrb_seamless.cuh -- the finish stage of the seamless streaming mode (DESIGN.md section 11).
//
// The default chain filters every chunk as if it were the whole signal.  The seamless mode filters
// the whole stream: the front ends (k_tc / k_main) and the IQ kernels run unchanged, chunk-local;
// everything chunk-local after them is replaced here.  A chunk's front-end outputs are the global
// ones times one phasor phi_{c,r} = exp(-2 pi i ((f_r N c) mod fs) / fs), so the kernels below
//
//   k_seam_edges   decode the head / end-window samples of every new chunk (kept for later calls)
//   k_seam_agg     chunk aggregates: the tile aggregates composed over a chunk (forward A, backward B)
//   k_seam_head    the stream's real start: odd extension and zi, forward state at sample 0
//   k_seam_fscan   forward modal state across chunks: affine scan with multiplier p^N per mode
//   k_seam_tail    the stream's real end: anticausal state after the last chunk and zeta
//                  (k_seam_head / tail run the chunk-boundary routines of k_fixup and k_finish, and
//                  k_seam_agg / y k_fixup's tile carries and outputs, sdrb_kernels.cuh)
//   k_seam_carry   per emitted chunk: carry-ins in its own frame (forward state, anticausal window
//                  over the next D chunks or the real end, zeta) and the fm halo y[k+1]
//   k_seam_y       per emitted chunk: tile carries and the decimated outputs, global frame
//   k_seam_demod   demodulation + output SOS from the chunk's zero state (the shared output stage of
//                  sdrb_outstage.cuh) and the chunk's end state; iq: y itself, (Re, Im) pairs;
//                  usb / lsb (SSB instance): the complex band-pass, its real part, a complex end state
//   k_seam_sscan   output SOS state across chunks: affine scan with the matrix A^M (real states), or
//                  e^{j Omega M} A^M (usb / lsb: complex states in the frame of each chunk's start)
//   k_seam_frame   response to the carried SOS state (usb / lsb: Re(e^{j Omega k} c A^k s_c)), framing
//
// tests/seamless_ref.py (SeamlessTwin) is the numpy twin of this decomposition.
#pragma once
#include <type_traits>
#include "sdrb_kernels.cuh"
#include "sdrb_outstage.cuh"

#define SEAM_NS 4           // output SOS state size in seamless mode (ellip(3): two sections); usb / lsb
                            // carry SEAM_NS complex states (echunk, sst and sos hold double2 then)

struct SeamDev {
    int D;                     // lookahead in chunks
    int nedge;                 // decoded samples kept per chunk: head (edge+1) + end window (nend); the
                               // stride holds a ragged last frame's longer window (max(edge+1, q-1))
    long long fs;
    const long long *step;     // [R] (f_r N) mod fs
    const double2 *PN;         // [D+1][8] p_i^(N j)
    double AM[SEAM_NS * SEAM_NS];   // A^M of the output cascade
    const double *CAM;         // [M][ns] c A^i
    // window buffers, slot = position in the window of unemitted chunks
    double2 *edges;            // [W][nedge]
    double2 *cagg;             // [W][R][16]   0..7 A (forward), 8..15 B (backward), global frame
    double2 *G;                // [W][R][8]    forward state at the chunk start, global frame
    double2 *cin;              // [W][R][24]   carry-ins in the chunk frame: Win0, Tn_end, zeta
    double2 *ybuf;             // [W][R][M+1]  decimated outputs (global frame) + halo
    double *echunk;            // [W][R][ns]   SOS end state of a chunk from a zero state (usb / lsb: ns complex)
    double *sst;               // [W][R][ns]   SOS state at the chunk start (after k_seam_sscan)
    double2 *fwd;              // [R][8]       forward state at the next new chunk
    double *sos;               // [R][ns]      SOS state at the next chunk to emit (usb / lsb: ns complex)
    double2 *endv;             // [R][16]      real end: 0..7 anticausal state, 8..15 zeta (global frame)
};

// the output SOS state of k_seam_sscan: real (fm / am) or complex (usb / lsb)
__device__ __forceinline__ double seam_add(double a, double b) { return a + b; }
__device__ __forceinline__ double2 seam_add(double2 a, double2 b) { return cadd(a, b); }
__device__ __forceinline__ double seam_rot(double2, double x) { return x; }            // real states: no phasor
__device__ __forceinline__ double2 seam_rot(double2 ph, double2 x) { return cmul(ph, x); }

__device__ __forceinline__ double2 seam_phasor(const SeamDev &sd, int r, long long g)
{
    const unsigned long long fs = (unsigned long long)sd.fs;
    const unsigned long long idx = ((unsigned long long)sd.step[r] * ((unsigned long long)g % fs)) % fs;
    double s, c;
    sincospi(-2.0 * ((double)idx / (double)sd.fs), &s, &c);
    return make_double2(c, s);
}

template <int ENC>
__global__ void __launch_bounds__(64)
k_seam_edges(const __grid_constant__ DevPlan pl, SeamDev sd, const uint8_t *__restrict__ raw, int slot0, int nch)
{
    const int c = blockIdx.x;
    if (c >= nch) return;
    const uint8_t *rawc = raw + (size_t)c * pl.N * pl.sb;
    double2 *e = sd.edges + (size_t)(slot0 + c) * sd.nedge;
    for (int j = threadIdx.x; j < pl.edge + 1 + pl.nend; j += blockDim.x) {
        const long n = j <= pl.edge ? j : (long)pl.ws + (j - pl.edge - 1);
        e[j] = decode_sample<ENC>(pl, rawc, n);
    }
}

// warp <-> (chunk, row); lanes 0..7 compose the forward tile aggregates, lanes 8..15 the backward ones;
// stored rotated into the global frame (phi_c A_c, phi_c B_c)
__global__ void __launch_bounds__(256)
k_seam_agg(const __grid_constant__ DevPlan pl, Scratch sc, SeamDev sd, int slot0, int nch, long long g0)
{
    const int lane = threadIdx.x & 31;
    const long item = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long)nch * pl.R || lane >= 16) return;
    const int c = slot0 + (int)(item / pl.R), r = (int)(item % pl.R), nt = pl.ntiles;
    const double2 a = tile_carries(pl, pl.T1 + (size_t)r * nt, sc.agg + ((size_t)c * pl.R + r) * nt * 16, lane & 7,
                                   lane < 8, make_double2(1.0, 0.0), make_double2(0.0, 0.0), [](size_t, double2) {});
    sd.cagg[((size_t)c * pl.R + r) * 16 + lane] = cmul(seam_phasor(sd, r, g0 + (c - slot0)), a);
}

// warp <-> row: forward state at sample 0 of the stream (sosfiltfilt's odd extension and zi)
__global__ void __launch_bounds__(32)
k_seam_head(const __grid_constant__ DevPlan pl, Scratch sc, SeamDev sd, int slot)
{
    __shared__ double2 s_ha[32];           // head extension (edge < 32)
    const int r = blockIdx.x, lane = threadIdx.x;
    const double2 *z = sd.edges + (size_t)slot * sd.nedge;
    const double2 off0 = sc.off_tile[(size_t)slot * (pl.ntiles + 1)];
    head_window(pl, r, lane <= pl.edge ? z[lane] : make_double2(0.0, 0.0), off0, s_ha, lane);
    double2 w = boundary_sums(pl, pl.pk, s_ha, pl.edge, s_ha, 0, lane).A;
    if (pl.correct_iq) w = cmul(cfma(pl.alpha[(size_t)r * 8 + (lane & 7)], off0, w), pl.binv[(size_t)r * 8 + (lane & 7)]);
    if (lane < 8) sd.fwd[(size_t)r * 8 + lane] = w;
}

// block <-> row, warp <-> mode, lane <-> contiguous run of chunks: G[c] = state before chunk c,
// G[c+1] = p^N G[c] + phi_c A_c, from the handle's forward state; the new state back into it
__global__ void __launch_bounds__(256)
k_seam_fscan(const __grid_constant__ DevPlan pl, SeamDev sd, int slot0, int nch)
{
    const int r = blockIdx.x, m = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double2 PN = sd.PN[8 + m];
    const int per = (nch + 31) / 32;
    const int c0 = min(nch, lane * per), c1 = min(nch, c0 + per);
    double2 a = make_double2(0.0, 0.0), mul = make_double2(1.0, 0.0);
    for (int c = c0; c < c1; c++) {
        a = cfma(PN, a, sd.cagg[((size_t)(slot0 + c) * pl.R + r) * 16 + m]);
        mul = cmul(mul, PN);
    }
    warp_affine_scan(mul, a, lane);
    const double2 st0 = sd.fwd[(size_t)r * 8 + m];
    double2 ea = shfl_up_c(a, 1), em = shfl_up_c(mul, 1);
    if (lane == 0) { ea = make_double2(0.0, 0.0); em = make_double2(1.0, 0.0); }
    double2 s = cfma(em, st0, ea);
    for (int c = c0; c < c1; c++) {
        sd.G[((size_t)(slot0 + c) * pl.R + r) * 8 + m] = s;
        s = cfma(PN, s, sd.cagg[((size_t)(slot0 + c) * pl.R + r) * 16 + m]);
    }
    if (lane == 31) sd.fwd[(size_t)r * 8 + m] = cfma(mul, st0, a);
}

// warp <-> row: the stream's real end (the last chunk sits in window slot `slot`, global index g)
__global__ void __launch_bounds__(32)
k_seam_tail(const __grid_constant__ DevPlan pl, Scratch sc, SeamDev sd, int slot, long long g)
{
    __shared__ double2 s_e[SDRB_NEDGE];    // end window (nend) + tail extension (edge)
    const int r = blockIdx.x, lane = threadIdx.x, m = lane & 7;
    const bool iq = pl.correct_iq != 0;
    const double2 *z = sd.edges + (size_t)slot * sd.nedge + pl.edge + 1;
    const double2 offE = sc.off_tile[(size_t)slot * (pl.ntiles + 1) + pl.ntiles];
    end_window(pl, r, [&](int j) { return z[j]; }, offE, s_e, lane);
    const double2 *seq = s_e + pl.nend - pl.rem;
    const int nseq = pl.rem + pl.edge;
    const BoundarySums bs = boundary_sums(pl, pl.pk, seq, 0, seq, nseq, lane);
    // at q*Mf: the true forward state, and the anticausal state into the T~ frame
    const double2 ph = seam_phasor(sd, r, g), sE = iq ? cmul(offE, pl.phE[r]) : make_double2(0.0, 0.0);
    double2 w = cmul(cconj(ph), sd.fwd[(size_t)r * 8 + m]);
    if (iq) w = csub(cmul(pl.beta[(size_t)r * 8 + m], w), cmul(pl.alpha[(size_t)r * 8 + m], sE));
    const double2 Tt = iq ? cmul(cfma(pl.alphaT[(size_t)r * 8 + m], sE, bs.B), pl.binvT[(size_t)r * 8 + m]) : bs.B;
    const double2 zeta = boundary_zeta(pl, pl.pk, seq, nseq, w, bs.C, lane);
    if (lane < 8) {
        sd.endv[(size_t)r * 16 + m] = cmul(ph, Tt);
        sd.endv[(size_t)r * 16 + 8 + m] = cmul(ph, zeta);
    }
    if (pl.rem) {       // a ragged last frame: the output at its partial block, as k_fixup's
        double2 v = cfma(pl.rho[m], w, cmul(pl.rho_p[m], bs.B));
        v = cfma(pl.bnd[(size_t)pl.Mf * 8 + m], zeta, v);
        for (int sft = 1; sft < 8; sft <<= 1) v = cadd(v, shfl_xor_c(v, sft));
        if (lane == 0)
            sd.ybuf[((size_t)slot * pl.R + r) * (pl.M + 1) + pl.Mf] =
                cmul(ph, make_double2(fma(pl.g0, seq[0].x, v.x), fma(pl.g0, seq[0].y, v.y)));
    }
}

// warp <-> row: a ragged last frame (its slot in `sd`) moves the real end to the last whole frame,
// so that k_seam_carry runs over the whole frames unchanged: the anticausal state crosses the
// frame's full blocks (pw[8..15] = p^(q Mf)) and takes its backward aggregate, zeta is referred to
// Lp samples earlier (pw[0..7] = p^Lp).
__global__ void __launch_bounds__(32)
k_seam_fold(SeamDev sd, const double2 *pw)
{
    const int r = blockIdx.x, m = threadIdx.x;
    if (m >= 8) return;
    double2 *e = sd.endv + (size_t)r * 16;
    e[m] = cfma(pw[8 + m], e[m], sd.cagg[(size_t)r * 16 + 8 + m]);
    e[8 + m] = cmul(pw[m], e[8 + m]);
}

// warp <-> (emitted chunk i, row), lane <-> mode.  Window slots 0..nwin-1 hold global chunks g0..;
// `end` = the real end of the stream is known (slot nwin-1 is the last chunk).
__global__ void __launch_bounds__(256)
k_seam_carry(const __grid_constant__ DevPlan pl, Scratch sc, SeamDev sd, int ne, int nwin, long long g0, int end)
{
    const int lane = threadIdx.x & 31;
    const long item = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long)ne * pl.R) return;
    const int i = (int)(item / pl.R), r = (int)(item % pl.R), m = lane & 7, R = pl.R, M = pl.M;
    const int dist = nwin - 1 - i;                       // chunks after this one in the window
    const bool known = end && dist <= sd.D, last = end && dist == 0;
    const int J = known ? dist : sd.D;
    const double2 PN1 = sd.PN[8 + m];
    double2 Tg = known ? sd.endv[(size_t)r * 16 + m] : make_double2(0.0, 0.0);
    for (int j = J; j >= 1; j--)
        Tg = cfma(PN1, Tg, sd.cagg[((size_t)(i + j) * R + r) * 16 + 8 + m]);
    double2 Zg = make_double2(0.0, 0.0);
    if (known) Zg = cmul(sd.PN[(size_t)dist * 8 + m], sd.endv[(size_t)r * 16 + 8 + m]);
    const double2 phc = cconj(seam_phasor(sd, r, g0 + i));
    if (lane < 8) {
        double2 *ci = sd.cin + ((size_t)i * R + r) * 24;
        ci[m] = cmul(phc, sd.G[((size_t)i * R + r) * 8 + m]);
        ci[8 + m] = cmul(phc, Tg);
        ci[16 + m] = cmul(phc, Zg);
    }
    if (last) return;
    // halo: block 0 of the next chunk, from this chunk's horizon
    double2 v = make_double2(0.0, 0.0);
    if (lane < 8) {
        v = cmul(pl.rb[(size_t)r * 8 + m], sd.G[((size_t)(i + 1) * R + r) * 8 + m]);
        v = cfma(pl.rbT[(size_t)r * 8 + m], Tg, v);
        if (known) v = cfma(pl.bnd[m], cmul(sd.PN[(size_t)(dist - 1) * 8 + m], sd.endv[(size_t)r * 16 + 8 + m]), v);
    }
#pragma unroll
    for (int o = 4; o >= 1; o >>= 1) v = cadd(v, shfl_xor_c(v, o));
    if (lane == 0) {
        const double2 z0 = sd.edges[(size_t)(i + 1) * sd.nedge];
        const double2 off1 = pl.correct_iq ? sc.off_tile[(size_t)i * (pl.ntiles + 1) + pl.ntiles] : make_double2(0.0, 0.0);
        const double2 loc = csub(cscale(pl.g0, z0), cmul(pl.gamma[r], off1));
        v = cfma(seam_phasor(sd, r, g0 + i + 1), loc, v);
        sd.ybuf[((size_t)i * R + r) * (M + 1) + M] = v;
    }
}

// warp <-> (emitted chunk, row): tile carries (lanes 0..7 forward, 8..15 backward) into sc.carry,
// then lane <-> block outputs, rotated into the global frame
__global__ void __launch_bounds__(256)
k_seam_y(const __grid_constant__ DevPlan pl, Scratch sc, SeamDev sd, int ne, int nwin, long long g0, int end)
{
    const int lane = threadIdx.x & 31;
    const long item = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long)ne * pl.R) return;
    const int i = (int)(item / pl.R), r = (int)(item % pl.R), nt = pl.ntiles, R = pl.R, M = pl.M, m = lane & 7;
    const double2 *ci = sd.cin + ((size_t)i * R + r) * 24;
    const double2 *T1 = pl.T1 + (size_t)r * nt;
    double2 *carry = sc.carry + ((size_t)i * R + r) * (nt + 1) * 16;
    auto keep = [&](size_t j, double2 v) { carry[j] = v; };
    if (lane < 16)
        tile_carries(pl, T1, sc.agg + ((size_t)i * R + r) * nt * 16, m, lane < 8,
                     (lane < 8 ? pl.beta : pl.betaT)[(size_t)r * 8 + m], ci[lane], keep);
    __syncwarp();
    const double2 ph = seam_phasor(sd, r, g0 + i);
    const bool has_z = end && nwin - 1 - i <= sd.D;     // zeta reaches this chunk
    double2 *y = sd.ybuf + ((size_t)i * R + r) * (M + 1);
    block_outputs(pl, r, sc.ypart + ((size_t)i * R + r) * pl.Mf, sc.off_tile + (size_t)i * (nt + 1), T1, carry,
                  ci + 16, has_z ? 0 : M, lane, 32, [&](int k, double2 v) { y[k] = cmul(ph, v); });
}

__device__ __forceinline__ double seam_demod_at(const double2 *y, int k, int M, bool last, int demod)
{
    if (demod != SDRB_FM) return demod_scalar(y[k], demod);
    if (last && k == M - 1) {
        if (M == 1) return pair_phase(y[1], y[0]);    // a one-output last frame: y[1] holds the output before it
        k = M - 2;
    }
    return pair_phase(y[k], y[k + 1]);
}

// warp <-> (emitted chunk, row), lane <-> segment of Lseg = ceil(M/32) outputs.  Without an output
// filter the demodulated values are framed and stored; with it the output stage runs the cascade
// from the chunk's zero state (sdrb_outstage.cuh) and the chunk's zero-state end state goes to
// echunk.  The response to the state carried from earlier chunks is k_seam_frame's.  The SSB
// instance runs the complex band-pass on y, its end state complex.  Rows of `out` are rs outputs
// long (W / M doubles each).  A ragged last frame comes in its own launch of the SHORT instance
// (M < 32 Lseg): its lanes stop at M (a short or empty segment only feeds the states of the lanes
// after it, whose outputs lie past M; its end state is not used, the stream ends there).
template <bool SSB, bool SHORT = false>
__global__ void __launch_bounds__(256)
k_seam_demod(const __grid_constant__ DevPlan pl, SeamDev sd, double *out, int ne, int nwin, int end, size_t rs)
{
    using T = std::conditional_t<SSB, double2, double>;
    const int lane = threadIdx.x & 31;
    const long item = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long)ne * pl.R) return;
    const int i = (int)(item / pl.R), r = (int)(item % pl.R), M = pl.M, lo = lane * pl.sos_Lseg;
    const bool last = end && i == nwin - 1;
    const double2 *y = sd.ybuf + ((size_t)i * pl.R + r) * (M + 1);
    double *o = out + (size_t)r * rs + (size_t)i * M;
    if (!SSB && pl.demod == SDRB_IQ) {     // rows of rs (Re, Im) pairs, no output low-pass
        double2 *o2 = reinterpret_cast<double2 *>(out) + (size_t)r * rs + (size_t)i * M;
        for (int k = lane; k < M; k += 32) frame_store(o2 + k, y[k], pl.be_out);
        return;
    }
    if (!SSB && pl.nsec_out == 0) {
        for (int k = lane; k < M; k += 32) frame_store(o + k, seam_demod_at(y, k, M, last, pl.demod), pl.be_out);
        return;
    }
    T st[SEAM_NS];
    sos_segments(
        pl, SEAM_NS / 2, lo, SHORT ? max(0, min(pl.sos_Lseg, M - lo)) : pl.sos_Lseg, lane,
        [&](int j) {
            if constexpr (SSB) return y[lo + j];
            else return seam_demod_at(y, lo + j, M, last, pl.demod);
        },
        [&](int j) -> double & { return o[lo + j]; }, st);
    if (lane == 31)
        for (int j = 0; j < SEAM_NS; j++) reinterpret_cast<T *>(sd.echunk)[((size_t)i * pl.R + r) * SEAM_NS + j] = st[j];
}

// one warp per row, lane <-> contiguous run of chunks: sst[c] = SOS state at the start of emitted
// chunk c, s[c+1] = A^M s[c] + echunk[c], from the handle's state; the new state back into it.
// T = double2 (usb / lsb): complex states in the frame of each chunk's first output, so the chunk
// map is e^{j Omega M} (A^M s[c] + echunk[c]); a composed map is a real matrix times a phasor.
template <typename T>
__global__ void __launch_bounds__(32)
k_seam_sscan(const __grid_constant__ DevPlan pl, SeamDev sd, int ne)
{
    constexpr bool CPX = std::is_same<T, double2>::value;
    const int r = blockIdx.x, lane = threadIdx.x;
    const int per = (ne + 31) / 32;
    const int c0 = min(ne, lane * per), c1 = min(ne, c0 + per);
    const T *ech = reinterpret_cast<const T *>(sd.echunk);
    T *sst = reinterpret_cast<T *>(sd.sst), *sos = reinterpret_cast<T *>(sd.sos);
    T a[SEAM_NS];
#pragma unroll
    for (int j = 0; j < SEAM_NS; j++) a[j] = zero_of<T>();
    double mm[SEAM_NS * SEAM_NS];
#pragma unroll
    for (int j = 0; j < SEAM_NS * SEAM_NS; j++) mm[j] = (j % (SEAM_NS + 1)) == 0 ? 1.0 : 0.0;
    double2 EM = make_double2(1.0, 0.0), ph = EM;   // chunk phasor e^{j Omega M}; phasor of the composed map
    if constexpr (CPX) EM = pl.ssb_rot[pl.M];
    auto matvec = [&](const double *A, const T *x, T *yv) {
#pragma unroll
        for (int p = 0; p < SEAM_NS; p++) {
            T acc = zero_of<T>();
#pragma unroll
            for (int q = 0; q < SEAM_NS; q++) acc = rfma(A[p * SEAM_NS + q], x[q], acc);
            yv[p] = acc;
        }
    };
    auto matmul = [&](const double *A, const double *B, double *C) {     // C = A B
#pragma unroll
        for (int p = 0; p < SEAM_NS; p++)
#pragma unroll
            for (int q = 0; q < SEAM_NS; q++) {
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < SEAM_NS; k++) acc = fma(A[p * SEAM_NS + k], B[k * SEAM_NS + q], acc);
                C[p * SEAM_NS + q] = acc;
            }
    };
    for (int c = c0; c < c1; c++) {
        T t[SEAM_NS];
        double t2[SEAM_NS * SEAM_NS];
        matvec(sd.AM, a, t);
        for (int j = 0; j < SEAM_NS; j++) a[j] = seam_rot(EM, seam_add(t[j], ech[((size_t)c * pl.R + r) * SEAM_NS + j]));
        matmul(sd.AM, mm, t2);
        for (int j = 0; j < SEAM_NS * SEAM_NS; j++) mm[j] = t2[j];
        if constexpr (CPX) ph = cmul(ph, EM);
    }
#pragma unroll
    for (int lv = 0; lv < 5; lv++) {
        T pa[SEAM_NS];
        double pm[SEAM_NS * SEAM_NS];
#pragma unroll
        for (int j = 0; j < SEAM_NS; j++) pa[j] = shfl_up_t(a[j], 1 << lv);
#pragma unroll
        for (int j = 0; j < SEAM_NS * SEAM_NS; j++) pm[j] = __shfl_up_sync(0xffffffffu, mm[j], 1 << lv);
        double2 pph = ph;
        if constexpr (CPX) pph = shfl_up_c(ph, 1 << lv);
        if (lane >= (1 << lv)) {
            T t[SEAM_NS];
            double t2[SEAM_NS * SEAM_NS];
            matvec(mm, pa, t);
            for (int j = 0; j < SEAM_NS; j++) a[j] = seam_add(a[j], seam_rot(ph, t[j]));
            matmul(mm, pm, t2);
            for (int j = 0; j < SEAM_NS * SEAM_NS; j++) mm[j] = t2[j];
            if constexpr (CPX) ph = cmul(ph, pph);
        }
    }
    T st0[SEAM_NS], ea[SEAM_NS];
    double em[SEAM_NS * SEAM_NS];
    for (int j = 0; j < SEAM_NS; j++) st0[j] = sos[(size_t)r * SEAM_NS + j];
#pragma unroll
    for (int j = 0; j < SEAM_NS; j++) ea[j] = shfl_up_t(a[j], 1);
#pragma unroll
    for (int j = 0; j < SEAM_NS * SEAM_NS; j++) em[j] = __shfl_up_sync(0xffffffffu, mm[j], 1);
    double2 eph = ph;
    if constexpr (CPX) eph = shfl_up_c(ph, 1);
    if (lane == 0) {
        for (int j = 0; j < SEAM_NS; j++) ea[j] = zero_of<T>();
        for (int j = 0; j < SEAM_NS * SEAM_NS; j++) em[j] = (j % (SEAM_NS + 1)) == 0 ? 1.0 : 0.0;
        eph = make_double2(1.0, 0.0);
    }
    T s[SEAM_NS];
    matvec(em, st0, s);
    for (int j = 0; j < SEAM_NS; j++) s[j] = seam_add(seam_rot(eph, s[j]), ea[j]);
    for (int c = c0; c < c1; c++) {
        T t[SEAM_NS];
        for (int j = 0; j < SEAM_NS; j++) sst[((size_t)c * pl.R + r) * SEAM_NS + j] = s[j];
        matvec(sd.AM, s, t);
        for (int j = 0; j < SEAM_NS; j++) s[j] = seam_rot(EM, seam_add(t[j], ech[((size_t)c * pl.R + r) * SEAM_NS + j]));
    }
    if (lane == 31) {
        T t[SEAM_NS];
        matvec(mm, st0, t);
        for (int j = 0; j < SEAM_NS; j++) sos[(size_t)r * SEAM_NS + j] = seam_add(seam_rot(ph, t[j]), a[j]);
    }
}

// thread <-> output: out += c A^k s[chunk], then framing; SSB: out += Re(e^{j Omega k} c A^k s[chunk]).
// Rows of rs outputs: M per chunk, the last chunk possibly shorter (a ragged last frame).
template <bool SSB>
__global__ void __launch_bounds__(256)
k_seam_frame(const __grid_constant__ DevPlan pl, SeamDev sd, double *out, size_t rs)
{
    using T = std::conditional_t<SSB, double2, double>;
    const size_t M = pl.M, total = (size_t)pl.R * rs;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / rs, rest = e % rs, i = rest / M, k = rest % M;
        const T *s = reinterpret_cast<const T *>(sd.sst) + (i * pl.R + r) * SEAM_NS;
        const double2 ph = SSB ? pl.ssb_rot[k] : make_double2(1.0, 0.0);
        frame_store(out + e, add_response<SEAM_NS>(out[e], sd.CAM + k * SEAM_NS, SEAM_NS, s, ph), pl.be_out);
    }
}
