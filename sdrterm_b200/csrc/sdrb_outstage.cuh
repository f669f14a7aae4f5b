// sdrb_outstage.cuh -- the output stage every finish path shares (k_finish, k_demod, k_seam_demod,
// k_seam_frame): the demodulator scalars, the framing store, and the output SOS cascade run by one
// warp over a row cut into 32 lane segments of Ls = sos_Lseg outputs.
//
// The cascade is scipy.signal.sosfilt's DF2T recurrence over out_sos from a zero state, state vector
// s (two states per section, ns = 2 nsec <= 8), s' = A s + b x, output c s + d x.  Lane l:
//   1. runs its segment from a zero state (sos_step): the zero-state outputs v and the end state e_l;
//   2. composes the segment maps s -> A^Ls s + e_l by an inclusive Kogge-Stone scan
//      (sos_lane_scan, AP[lv] = (A^Ls)^(2^lv)): it then holds the state after segment l;
//   3. takes lane l-1's state as the state entering its segment and adds its response c A^j s_in
//      (CA[j] = c A^j) to output j of the segment (add_response).
// usb / lsb run the same cascade with complex states in the Weaver frame: u[k] = y[k] e^{-j Omega k}
// through the real prototype, Re and Im alike, keeping Re(e^{j Omega k} v[k]) (DESIGN.md section 13).
#pragma once
#include <type_traits>
#include "../../include/sdrterm_b200.h"
#include "sdrb_device.cuh"

// ---------------------------------------------------------------- demodulator scalars, framing
// fm: the phase of a conj(b) for the output pair (a, b) (demodulation.py:25-38)
__device__ __forceinline__ double pair_phase(double2 a, double2 b)
{
    return atan2(fma(a.y, b.x, -a.x * b.y), fma(a.x, b.x, a.y * b.y));
}

// am: abs(square(z)) (demodulation.py:41-48); re; im
__device__ __forceinline__ double demod_scalar(double2 a, int demod)
{
    if (demod == SDRB_AM) return hypot(fma(a.x, a.x, -a.y * a.y), 2.0 * a.x * a.y);
    return demod == SDRB_RE ? a.x : a.y;
}

__device__ __forceinline__ double bswap_double(double v)
{
    unsigned long long u = (unsigned long long)__double_as_longlong(v);
    uint32_t lo = (uint32_t)u, hi = (uint32_t)(u >> 32);
    u = ((unsigned long long)__byte_perm(lo, 0, 0x0123) << 32) | __byte_perm(hi, 0, 0x0123);
    return __longlong_as_double((long long)u);
}

// one output double, or one iq (Re, Im) pair, native or big-endian per double
__device__ __forceinline__ void frame_store(double *o, double v, int be) { *o = be ? bswap_double(v) : v; }
__device__ __forceinline__ void frame_store(double2 *o, double2 v, int be)
{
    if (be) v = make_double2(bswap_double(v.x), bswap_double(v.y));
    *o = v;
}

// ---------------------------------------------------------------- real or complex cascade states
template <typename T> __device__ __forceinline__ T zero_of();
template <> __device__ __forceinline__ double zero_of<double>() { return 0.0; }
template <> __device__ __forceinline__ double2 zero_of<double2>() { return make_double2(0.0, 0.0); }
__device__ __forceinline__ double rfma(double a, double x, double acc) { return fma(a, x, acc); }
__device__ __forceinline__ double2 rfma(double a, double2 x, double2 acc) { return make_double2(fma(a, x.x, acc.x), fma(a, x.y, acc.y)); }
__device__ __forceinline__ double shfl_up_t(double v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
__device__ __forceinline__ double2 shfl_up_t(double2 v, int d) { return shfl_up_c(v, d); }

// ---------------------------------------------------------------- the cascade
// One output of the DF2T cascade (nsec <= NS/2 sections; st[2s], st[2s+1] = the states of section s).
// Real: every product and sum rounded on its own, as the fused path has always computed it.
template <int NS>
__device__ __forceinline__ double sos_step(const double *sos, int nsec, double (&st)[NS], double x)
{
#pragma unroll
    for (int s = 0; s < NS / 2; s++) {
        if (s < nsec) {
            const double *cf = sos + 6 * s;
            const double xn = __dadd_rn(__dmul_rn(cf[0], x), st[2 * s]);
            st[2 * s] = __dadd_rn(__dadd_rn(__dmul_rn(cf[1], x), -__dmul_rn(cf[4], xn)), st[2 * s + 1]);
            st[2 * s + 1] = __dadd_rn(__dmul_rn(cf[2], x), -__dmul_rn(cf[5], xn));
            x = xn;
        }
    }
    return x;
}
// Complex (the Weaver frame): the real prototype on Re and Im alike, fused.
template <int NS>
__device__ __forceinline__ double2 sos_step(const double *sos, int nsec, double2 (&st)[NS], double2 x)
{
#pragma unroll
    for (int s = 0; s < NS / 2; s++) {
        if (s < nsec) {
            const double *cf = sos + 6 * s;
            const double2 xn = make_double2(fma(cf[0], x.x, st[2 * s].x), fma(cf[0], x.y, st[2 * s].y));
            st[2 * s] = make_double2(fma(cf[1], x.x, fma(-cf[4], xn.x, st[2 * s + 1].x)),
                                     fma(cf[1], x.y, fma(-cf[4], xn.y, st[2 * s + 1].y)));
            st[2 * s + 1] = make_double2(fma(cf[2], x.x, -cf[5] * xn.x), fma(cf[2], x.y, -cf[5] * xn.y));
            x = xn;
        }
    }
    return x;
}

// Inclusive Kogge-Stone scan of the 32 lane-segment maps s -> A^Ls s + st_lane (ns states,
// AP = [5][ns][ns]); afterwards lane l holds the state after segment l from a zero state at the start
// of segment 0.  Highest state index innermost in every FMA chain.
template <int NS, typename T>
__device__ __forceinline__ void sos_lane_scan(const double *AP, int ns, T (&st)[NS], int lane)
{
#pragma unroll
    for (int lv = 0; lv < 5; lv++) {
        T o[NS];
#pragma unroll
        for (int b = 0; b < NS; b++)
            if (b < ns) o[b] = shfl_up_t(st[b], 1 << lv);
        if (lane >= (1 << lv)) {
            const double *A = AP + lv * ns * ns;
#pragma unroll
            for (int a = 0; a < NS; a++) {
                if (a < ns) {
                    T acc = st[a];
#pragma unroll
                    for (int b = NS - 1; b >= 0; b--)
                        if (b < ns) acc = rfma(A[a * ns + b], o[b], acc);
                    st[a] = acc;
                }
            }
        }
    }
}

// v plus the kept part of the response c A^j s to a state s (ca = c A^j, ns states): real states
// v + c A^j s, one FMA chain from v, highest state index innermost; usb / lsb v + Re(ph c A^j s)
// with ph = e^{j Omega k}.
template <int NS>
__device__ __forceinline__ double add_response(double v, const double *ca, int ns, const double *s, double2)
{
#pragma unroll
    for (int b = NS - 1; b >= 0; b--)
        if (b < ns) v = fma(ca[b], s[b], v);
    return v;
}
template <int NS>
__device__ __forceinline__ double add_response(double v, const double *ca, int ns, const double2 *s, double2 ph)
{
    double2 w = make_double2(0.0, 0.0);
#pragma unroll
    for (int b = NS - 1; b >= 0; b--)
        if (b < ns) w = rfma(ca[b], s[b], w);
    return fma(ph.x, w.x, fma(-ph.y, w.y, v));
}

// The output cascade on lane segment `lane` of a row: n outputs (the row's outputs lo .. lo+n-1; n
// < Ls only where the row ends), steps 1-3 above.  in(j) gives the cascade input of output lo+j (a
// double, or y itself for usb / lsb: T = double2), out(j) a double& to its slot, written in step 1
// and updated in step 3, both in ascending j.  st returns the lane's inclusive state: on lane 31 the
// state after the row from a zero start (seamless mode carries it into the next chunk).
template <int NS, typename T, typename In, typename Out>
__device__ __forceinline__ void sos_segments(const DevPlan &pl, int nsec, int lo, int n, int lane, In in, Out out,
                                             T (&st)[NS])
{
    constexpr bool CPX = std::is_same<T, double2>::value;
    const int ns = 2 * nsec;
    double2 e1 = make_double2(1.0, 0.0), r0 = e1;           // usb / lsb: e^{j Omega}, e^{j Omega lo}
    if constexpr (CPX) { e1 = pl.ssb_rot[1]; r0 = pl.ssb_rot[lo]; }
    double2 ph = r0;
#pragma unroll
    for (int a = 0; a < NS; a++) st[a] = zero_of<T>();
#pragma unroll (CPX ? 2 : 4)
    for (int j = 0; j < n; j++) {
        if constexpr (CPX) {
            const double2 v = sos_step(pl.out_sos, nsec, st, cmul(in(j), cconj(ph)));
            out(j) = fma(ph.x, v.x, -ph.y * v.y);
            ph = cmul(ph, e1);
        } else {
            out(j) = sos_step(pl.out_sos, nsec, st, in(j));
        }
    }
    sos_lane_scan(pl.sos_AP, ns, st, lane);
    T si[NS];
#pragma unroll
    for (int a = 0; a < NS; a++) {
        si[a] = shfl_up_t(st[a], 1);
        if (lane == 0) si[a] = zero_of<T>();
    }
    ph = r0;
#pragma unroll (CPX ? 2 : 4)
    for (int j = 0; j < n; j++) {
        double &o = out(j);
        o = add_response<NS>(o, pl.sos_CA + (size_t)j * ns, ns, si, ph);
        if constexpr (CPX) ph = cmul(ph, e1);
    }
}
