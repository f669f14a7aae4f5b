// sdrb_tc.cuh -- k_tc: the block front end on the 5th-generation tensor cores (tcgen05, sm_100a).
//
// Every per-block quantity of the chain -- decode, byte order, NCO, the 16 modal block sums, the
// IQ-EMA aggregates AND the part of each decimated output that is local to its neighbourhood -- is
// a real-linear functional of the raw integer samples, i.e. one row of a coefficient matrix applied
// to the raw bytes.  sdrterm_b200/plan.py (build_tc) rounds the coefficients to 40-bit fixed point
// and cuts them into 5 balanced base-256 digits, so that
//
//     D[superblock, 5*o + t] = sum_k  rawbyte[superblock, k] * digit[o, t, k]     (int8 x int8 -> int32)
//
// is an EXACT integer GEMM: A = the raw stream itself, viewed as [super-blocks][K] bytes (a
// super-block = 2 consecutive blocks of q samples, K = 256 or 512 bytes) and brought in by TMA
// (128B swizzle) without ever being decoded; B = the digit matrix of this CTA's row of the VFO
// bank, resident in shared memory; D in tensor memory (2 stages x 208 columns).  Outputs per
// super-block: F~_i, G~_i (8 + 8 complex modal sums over the 2q samples), E_a, E_ab (IQ-EMA
// aggregates after q and 2q samples), yl_a, yl_b (the two block outputs' super-block-local part).
// The samples are NOT IQ-corrected here: the corrector is decoupled from the modal sums
// (DESIGN.md 3.3) and enters as one term per output, -gamma * (rotated offset).
//
// Warp roles (512 threads, one CTA per SM, persistent over MMA tiles of 128 super-blocks; a CTA
// serves one row r of the VFO bank, blockIdx.x % R):
//   warp 0      TMA producer (one lane): a ring of 16 KB stages, one 128-byte K slab of a tile each
//   warp 1      TMEM allocation; tcgen05.mma issue (one lane): 4 MMAs (K = 32) per slab; the MMA's
//               own completion frees the slab (tcgen05.commit) and, after the last slab of a tile,
//               signals the epilogue
//   warps 2-3   sign fix-up: XOR 0x80 into the bytes that are not the signed top byte, so that
//               every byte is a valid two's-complement int8 operand (the constant this removes is
//               added back as cst[o])
//   warps 4-15  epilogue: warp = 4 + 4*group + quarter; the three groups take the MMA tiles
//               round-robin (an epilogue pass is a long chain of dependent FP64 operations: three
//               tiles in flight per SM hide it, the two TMEM stages are free again as soon as a
//               group has read its columns).  `quarter` (= warp % 4) is the TMEM lane
//               quarter = 32 super-blocks (lane <-> super-block) = 2 tiles of 32 blocks:
//               digit columns -> FP64 (exact up to one rounding), tile-local IQ offsets, forward and
//               backward modal scans in the rotating frame (lane = (segment of 8 super-blocks,
//               mode) through one shared-memory transpose each way), the two block outputs of
//               every super-block, tile aggregates for k_finish
//
// Reference behaviour reproduced: src/misc/read_file.py:100-103, src/dsp/demodulation.py:71-79,
// the block form of scipy.signal.decimate (src/dsp/dsp_processor.py:147).  tests/emulator.py
// (emu_main_tc) is the numpy twin.
#pragma once
#include <cuda.h>
#include "sdrb_kernels.cuh"

#define TC_NOUT 40                     // fixed-point outputs per row: 16 F, 16 G, 4 E, 4 yl
#define TC_NCOL 5                      // digit columns per output
#define TC_NPAD 208                    // GEMM N per row (200 + 8 unit-coefficient x0 columns)
#define TC_X0COL 200
#define TC_MAX_R 32                    // rows of the VFO bank this kernel takes
#define TC_THREADS 512
#define TC_EPI_WARPS 12
#define TC_EPI_GROUPS 3                // groups of 4 epilogue warps take the MMA tiles round-robin
#define TC_XS 33                       // exchange-buffer row stride in double2
#define TC_STAGES 2                    // TMEM accumulator stages (256 columns apart)
#define TC_MAX_ASTAGES 8               // shared-memory A ring (TMA -> sign fix-up -> MMA)
#define TC_REGION_BYTES 16384          // 128 rows x 128 bytes, one SWIZZLE_128B operand slab
#define TC_NROWC 200                   // complex constants per row (plan.py RC_* layout)
#define TC_RC_CA 0
#define TC_RC_CB 8
#define TC_RC_DA 16
#define TC_RC_DB 24
#define TC_RC_GAM 32
#define TC_RC_GAMQ 33
#define TC_RC_AGGF 34
#define TC_RC_ROT 36
#define TC_RC_POW 52

struct TcDev {
    int K, isz, nregion, nstage;
    uint32_t xor_word;                 // XOR pattern of 4 consecutive stream bytes
    uint32_t idesc;                    // tcgen05 instruction descriptor (i8 x i8 -> s32, M=128, N=208)
    double scale, scale16;             // 2^-S, 2^(16-S): outputs 0..35
    double scale_yl, scale16_yl;       // the same for the local outputs 36..39
    const double2 *rowc;               // [R][TC_NROWC]
    const double *cstb;                // [R][TC_NOUT + 4] response to the constant the XOR removed, minus
                                       // the 2^52 + 2^31 bias of the low digit pair (x0: minus the bias itself)
};

__host__ __device__ inline size_t tc_b_bytes(int nregion) { return (size_t)nregion * TC_NPAD * 128; }
__host__ __device__ inline size_t tc_fixed_bytes(int nregion)
{
    size_t b = tc_b_bytes(nregion);                                   // B slabs
    b += (size_t)TC_EPI_WARPS * 8 * TC_XS * sizeof(double2);          // xs[8 modes][33] per epilogue warp
    b += TC_NROWC * sizeof(double2) + 48 * sizeof(double);            // row constants, cstb
    b += 32 * sizeof(unsigned long long);                             // mbarriers
    return b + 1024;                                                  // alignment slack
}
__host__ __device__ inline size_t tc_smem_bytes(int nregion, int nstage)
{
    return tc_fixed_bytes(nregion) + (size_t)nstage * TC_REGION_BYTES;
}

// ------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t cnt)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(cnt));
}
__device__ __forceinline__ void mbar_arrive(uint32_t a)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t a, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes or
// the hint (ns) expires, instead of the warp burning issue slots in a spin loop.
__device__ __forceinline__ bool mbar_try(uint32_t a, uint32_t parity, uint32_t hint_ns)
{
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(a), "r"(parity), "r"(hint_ns) : "memory");
    return ok != 0;
}
// Bounded waits: a protocol error traps (and surfaces as a CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity)
{
    uint32_t n = 0;
    while (!mbar_try(a, parity, 20000u))
        if (++n > (1u << 22)) __trap();
}
__device__ __forceinline__ void mbar_wait_sleep(uint32_t a, uint32_t parity)
{
    uint32_t n = 0;
    while (!mbar_try(a, parity, 100000u))
        if (++n > (1u << 20)) __trap();
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int x, int y, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(bar) : "memory");
}
// L2 policies: the raw stream is read exactly once (evict first), while ypart / agg are read back
// by k_finish a moment later (evict last) -- 100 MB of intermediates then survive in the 126 MB L2
// instead of being flushed by the 1 GiB of raw bytes streaming past them.
#define TC_L2_EVICT_FIRST 0x12F0000000000000ull
#define TC_L2_EVICT_LAST 0x14F0000000000000ull
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap *map, int x, int y, uint32_t bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(bar), "l"(policy) : "memory");
}
__device__ __forceinline__ void st_keep_l2(double2 *p, double2 v)
{
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(v.x), "d"(v.y), "l"(TC_L2_EVICT_LAST) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory operand descriptor (8-row atoms of 128 bytes, 1024 B apart).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr)
{
    uint64_t d = (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;                  // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;        // stride byte offset between 8-row atoms
    d |= (uint64_t)1 << 46;                  // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                  // SWIZZLE_128B
    return d;
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t *r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t *r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t *r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t *r)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
}
// 20 consecutive columns = the digit columns of 4 outputs (2 complex values)
__device__ __forceinline__ void tmem_ld20(uint32_t taddr, uint32_t *r)
{
    tmem_ld16(taddr, r);
    tmem_ld4(taddr + 16, r + 16);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Exact int64 -> double for |v| < 2^51 without the slow I2F.F64 path: bias into the mantissa of
// 1.5 * 2^52 and subtract it again.
__device__ __forceinline__ double i64_to_double(long long v)
{
    return __longlong_as_double(v + 0x4338000000000000LL) - 6755399441055744.0;
}
// int32 -> 2^52 + 2^31 + v as a double (exact); the caller folds the bias into its constant.
__device__ __forceinline__ double i32_biased(int v)
{
    return __hiloint2double(0x43300000, v ^ 0x80000000);
}
#define TC_BIAS32 4503601774854144.0      // 2^52 + 2^31

// Digit columns c[0..5) (most significant first, weight 256 per step) -> value * 2^-S + cst.
// Column sums are bounded by 128 * (L1 norm of the digit column) < 2^31 / 257 (checked when the
// tables are built), so the pairs c1*256 + c2 and c3*256 + c4 fit 32 bits; the upper three columns
// are joined by one wide multiply-add and converted through the 2^52 bias, the low pair rides on
// the bias of a single FMA whose constant `cstb` = cst - (2^52 + 2^31) * 2^-S already removes it.
__device__ __forceinline__ double tc_combine(const uint32_t *c, double s16, double s1, double cstb)
{
    const int mid = (int)c[1] * 256 + (int)c[2];
    const int lo = (int)c[3] * 256 + (int)c[4];
    const long long hi = (long long)(int)c[0] * 65536 + (long long)mid;
    return fma(i64_to_double(hi), s16, fma(i32_biased(lo), s1, cstb));
}

#define TC_DBG(sc, it, ev) do { if ((sc).dbg && blockIdx.x == 0 && (it) < 32) (sc).dbg[(it) * 16 + (ev)] = clock64(); } while (0)

struct TcShared {
    unsigned char *sB, *sA;
    double2 *sXS, *sRow;
    double *sCst;
    uint32_t bar0;
};
enum { TCB_FULL_A = 0, TCB_XORED = 1, TCB_A_FREE = 2, TCB_MISC = 3 };   // MISC: 2,3 TMEM_FREE; 4..6 MMA_DONE; 7 BFULL
__device__ __forceinline__ uint32_t tc_bar(uint32_t bar0, int kind, int s)
{
    return bar0 + 8u * (uint32_t)(kind * TC_MAX_ASTAGES + s);
}

// Two complex values (4 outputs o0..o0+3) from 20 digit columns.
__device__ __forceinline__ void tc_combine2(const uint32_t *c, const double *cst, int o0, double s16, double s1, double2 *out)
{
#pragma unroll
    for (int m = 0; m < 2; m++) {
        const double2 cs = *reinterpret_cast<const double2 *>(cst + o0 + 2 * m);
        out[m].x = tc_combine(c + 10 * m, s16, s1, cs.x);
        out[m].y = tc_combine(c + 10 * m + 5, s16, s1, cs.y);
    }
}

// ------------------------------------------------------------------------------------- epilogue
// One warp, one quarter of an MMA tile: lane <-> super-block (2 blocks), lanes 0..15 and 16..31
// are two tiles of 32 blocks.  BACK = false: forward scan of the 8 modal sums in xs (state entering
// every super-block), BACK = true: backward scan (state above every super-block); the tile
// aggregates go to `agg`, the scan states are left in xs (lane <-> super-block view) for the
// output dots.
template <bool BACK>
__device__ __forceinline__ void tc_scan(double2 *xs, const double2 *sRow, int lane, double2 *agg_tile)
{
    const int mode = lane & 7, seg = lane >> 3;
    double2 *xsp = xs + mode * TC_XS + seg * 8;
    const double2 *pw = sRow + TC_RC_POW + ((BACK ? 8 : 0) + mode) * 9;
    const double2 Pm = pw[1];
    // positions in scan order: k = 0..7 (forward: j = k, backward: j = 7 - k); two independent
    // chains over k = 0..3 and k = 4..7 halve the dependent-FMA latency, the second half then
    // receives the first half's total like a carry
    double2 v[8], loc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = xsp[BACK ? 7 - k : k];
    double2 sA = make_double2(0.0, 0.0), sB = sA;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        loc[k] = sA;     sA = cfma(Pm, sA, v[k]);               // exclusive: state before this super-block
        loc[4 + k] = sB; sB = cfma(Pm, sB, v[4 + k]);
    }
    const double2 st = cfma(pw[4], sA, sB);                     // segment total
    // carry between the two segments of a tile (segments 0,1 = tile 0; 2,3 = tile 1)
    const bool second = BACK ? !(seg & 1) : (seg & 1);          // the segment that receives a carry
    const double2 other = shfl_c(st, lane ^ 8);
    const double2 cin = second ? other : make_double2(0.0, 0.0);
    const double2 cinB = cfma(pw[4], cin, sA);                  // what enters the second half-chain
    if (second) {
        const double2 tot = cfma(pw[8], cin, st);
        if (BACK) st_keep_l2(agg_tile + 8 + mode, tot);
        else st_keep_l2(agg_tile + mode, cmul(sRow[TC_RC_AGGF], tot));
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        xsp[BACK ? 7 - k : k] = cfma(pw[k], cin, loc[k]);
        xsp[BACK ? 3 - k : 4 + k] = cfma(pw[k], cinB, loc[4 + k]);
    }
}

template <bool IQ>
__device__ __forceinline__ void tc_epilogue(const DevPlan &pl, const TcDev &tc, const Scratch &sc, const TcShared &sh,
                                            uint32_t tmem_base, int e, int lane, int r, int slot, int nslots,
                                            int my_iters, int total_wtiles)
{
    const int qd = e & 3, grp = e >> 2;                         // TMEM lane quarter, epilogue group
    double2 *xs = sh.sXS + (size_t)e * 8 * TC_XS;
    double2 *xsl = xs + lane;                                   // lane <-> super-block view
    const double2 *sRow = sh.sRow;
    const double *sCst = sh.sCst;
    const uint32_t bar_done = tc_bar(sh.bar0, TCB_MISC, 4 + grp);
    const int l16 = lane & 15;
    const double s16 = tc.scale16, s1 = tc.scale;

    for (int it = grp, kk = 0; it < my_iters; it += TC_EPI_GROUPS, kk++) {
        const int g = it & 1;                                   // TMEM accumulator stage of this tile
        const uint32_t bar_free = tc_bar(sh.bar0, TCB_MISC, 2 + g);
        const uint32_t trow = tmem_base + ((uint32_t)(32 * qd) << 16) + (uint32_t)(g * 256);
        const int mt = slot + it * nslots;
        const int wt = 4 * mt + qd;                             // warp-tile: 32 super-blocks = 2 tiles
        if (lane == 0) mbar_wait(bar_done, kk & 1);
        __syncwarp();
        tc_fence_after();
        if (e == 0 && lane == 0) TC_DBG(sc, it, 5);
        if (wt >= total_wtiles) {
            if (lane == 0) mbar_arrive(bar_free);
            continue;
        }
        const int gt = 2 * wt + (lane >> 4);
        const int chunk = gt / pl.ntiles, t = gt - chunk * pl.ntiles;

        // ---- TMEM -> registers -> FP64, 20 columns (2 complex values) at a time; the load of the
        //      next 20 is in flight while the current ones are recombined.  The IQ aggregates come
        //      first so that their warp scan overlaps the remaining loads.
        uint32_t ca[20], cb[20];
        double2 gq[8], ev[2], yl[2], v2[2];
        tmem_ld20(trow + 160, ca);                              // E_a, E_ab
        tmem_ld_wait();
        tmem_ld20(trow, cb);                                    // F 0,1
        tc_combine2(ca, sCst, 32, s16, s1, ev);
        // IQ: tile-local offsets at the two block starts of every super-block (zero at the tile
        // start), tile aggregate
        double2 exa = make_double2(0.0, 0.0), exb = exa;
        if (IQ) {
            double2 inc = make_double2(pl.Liq * ev[1].x, pl.Liq * ev[1].y);
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const double2 tt = shfl_up_c(inc, 1 << i);
                if (l16 >= (1 << i)) { inc.x = fma(pl.lamq_pow[i + 1], tt.x, inc.x); inc.y = fma(pl.lamq_pow[i + 1], tt.y, inc.y); }
            }
            exa = shfl_up_c(inc, 1);
            if (l16 == 0) exa = make_double2(0.0, 0.0);
            if (l16 == 15 && r == 0) sc.tile_agg[(size_t)chunk * pl.ntiles + t] = inc;
            exb = make_double2(fma(pl.lam_q, exa.x, pl.Liq * ev[0].x), fma(pl.lam_q, exa.y, pl.Liq * ev[0].y));
        }
#define TC_STEP(CUR, NXT, NEXTCOL, O0, DST)                                                   \
        tmem_ld_wait();                                                                       \
        if ((NEXTCOL) >= 0) tmem_ld20(trow + (NEXTCOL), NXT);                                 \
        tc_combine2(CUR, sCst, O0, s16, s1, DST);
        TC_STEP(cb, ca, 20, 0, v2)   xsl[0 * TC_XS] = v2[0]; xsl[1 * TC_XS] = v2[1];          // F 0,1
        TC_STEP(ca, cb, 40, 4, v2)   xsl[2 * TC_XS] = v2[0]; xsl[3 * TC_XS] = v2[1];          // F 2,3
        TC_STEP(cb, ca, 60, 8, v2)   xsl[4 * TC_XS] = v2[0]; xsl[5 * TC_XS] = v2[1];          // F 4,5
        TC_STEP(ca, cb, 80, 12, v2)  xsl[6 * TC_XS] = v2[0]; xsl[7 * TC_XS] = v2[1];          // F 6,7
        TC_STEP(cb, ca, 100, 16, gq)                                                          // G 0,1
        TC_STEP(ca, cb, 120, 20, gq + 2)
        TC_STEP(cb, ca, 140, 24, gq + 4)
        TC_STEP(ca, cb, 180, 28, gq + 6)                                                      // next: yl_a, yl_b
        uint32_t cx[8];
        if (sc.x0) tmem_ld8(trow + TC_X0COL, cx);
        tmem_ld_wait();
#undef TC_STEP
        tc_combine2(cb, sCst, 36, tc.scale16_yl, tc.scale_yl, yl);   // the local outputs have their own finer scale
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_free);
        if (e == 0 && lane == 0) TC_DBG(sc, it, 6);

        const size_t obase = ((size_t)chunk * pl.R + r) * pl.Mf + (size_t)t * SDRB_TB + 2 * l16;
        if (sc.x0) {                                            // exact first samples (parity tests)
            int xr0, xi0, xr1, xi1;
            if (tc.isz == 2) {
                xr0 = (int)cx[0] * 256 + (int)cx[1]; xi0 = (int)cx[2] * 256 + (int)cx[3];
                xr1 = (int)cx[4] * 256 + (int)cx[5]; xi1 = (int)cx[6] * 256 + (int)cx[7];
            } else {
                xr0 = (int)cx[0]; xi0 = (int)cx[1]; xr1 = (int)cx[2]; xi1 = (int)cx[3];
            }
            sc.x0[obase] = make_double2(i32_biased(xr0) + sCst[40], i32_biased(xi0) + sCst[41]);
            sc.x0[obase + 1] = make_double2(i32_biased(xr1) + sCst[42], i32_biased(xi1) + sCst[43]);
        }

        if (e == 0 && lane == 0) TC_DBG(sc, it, 8);
        double2 *agg_tile = sc.agg + (((size_t)chunk * pl.R + r) * pl.ntiles + t) * 16;
        // ---- forward scan (the F sums were parked above), dots with the forward states
        __syncwarp();
        tc_scan<false>(xs, sRow, lane, agg_tile);
        __syncwarp();
        if (e == 0 && lane == 0) TC_DBG(sc, it, 9);
        // four independent accumulation chains per direction (the dependent-FMA latency, not the
        // FMA count, is what an epilogue warp waits for)
        double2 ya = yl[0], yb = yl[1], ya2 = make_double2(0.0, 0.0), yb2 = ya2;
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
            const double2 a = xsl[i * TC_XS], a2 = xsl[(i + 1) * TC_XS];
            ya = cfma(sRow[TC_RC_CA + i], a, ya);
            yb = cfma(sRow[TC_RC_DA + i], a, yb);
            ya2 = cfma(sRow[TC_RC_CA + i + 1], a2, ya2);
            yb2 = cfma(sRow[TC_RC_DA + i + 1], a2, yb2);
        }
        __syncwarp();
        if (e == 0 && lane == 0) TC_DBG(sc, it, 10);
        // ---- backward scan, dots with the backward states
#pragma unroll
        for (int m = 0; m < 8; m++) xsl[m * TC_XS] = gq[m];
        __syncwarp();
        tc_scan<true>(xs, sRow, lane, agg_tile);
        __syncwarp();
        if (e == 0 && lane == 0) TC_DBG(sc, it, 11);
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
            const double2 b = xsl[i * TC_XS], b2 = xsl[(i + 1) * TC_XS];
            ya = cfma(sRow[TC_RC_CB + i], b, ya);
            yb = cfma(sRow[TC_RC_DB + i], b, yb);
            ya2 = cfma(sRow[TC_RC_CB + i + 1], b2, ya2);
            yb2 = cfma(sRow[TC_RC_DB + i + 1], b2, yb2);
        }
        ya = cadd(ya, ya2); yb = cadd(yb, yb2);
        __syncwarp();
        if (IQ) {
            const double2 gm = sRow[TC_RC_GAM], gq2 = sRow[TC_RC_GAMQ];
            ya = cfma(make_double2(-gm.x, -gm.y), exa, ya);
            yb = cfma(make_double2(-gq2.x, -gq2.y), exb, yb);
        }
        const double2 rot = sRow[TC_RC_ROT + l16];
        double2 *yp = sc.ypart + obase;
        st_keep_l2(yp, cmul(rot, ya));
        st_keep_l2(yp + 1, cmul(rot, yb));
        if (e == 0 && lane == 0) TC_DBG(sc, it, 7);
    }
}

template <bool IQ>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc(const __grid_constant__ DevPlan pl, const __grid_constant__ TcDev tc, const __grid_constant__ Scratch sc,
     const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
     int n_mtiles, int total_wtiles)
{
    extern __shared__ unsigned char smem_dyn[];
    // keep the shared address space visible to the compiler: offset the array, do not re-cast
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nreg = tc.nregion, nstage = tc.nstage;
    TcShared sh;
    sh.sB = smem;
    sh.sA = sh.sB + tc_b_bytes(nreg);
    sh.sXS = reinterpret_cast<double2 *>(sh.sA + (size_t)nstage * TC_REGION_BYTES);
    sh.sRow = sh.sXS + (size_t)TC_EPI_WARPS * 8 * TC_XS;
    sh.sCst = reinterpret_cast<double *>(sh.sRow + TC_NROWC);
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(sh.sCst + 48);
    __shared__ uint32_t tmem_base_s;
    const uint32_t bar0 = smem_u32(bars);
    sh.bar0 = bar0;
    unsigned char *sA = sh.sA, *sB = sh.sB;

    // one row of the bank per CTA; the CTAs of a row share its MMA tiles round-robin
    const int r = (int)blockIdx.x % pl.R;
    const int slot = (int)blockIdx.x / pl.R, nslots = (int)gridDim.x / pl.R;

    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; s++) {
            mbar_init(tc_bar(bar0, TCB_FULL_A, s), 1);
            mbar_init(tc_bar(bar0, TCB_XORED, s), 2);
            mbar_init(tc_bar(bar0, TCB_A_FREE, s), 1);
        }
        for (int s = 0; s < TC_STAGES; s++)
            mbar_init(tc_bar(bar0, TCB_MISC, 2 + s), 4);        // TMEM_FREE: the 4 warps that read the stage
        for (int s = 0; s < TC_EPI_GROUPS; s++)
            mbar_init(tc_bar(bar0, TCB_MISC, 4 + s), 1);        // MMA_DONE, one per epilogue group
        mbar_init(tc_bar(bar0, TCB_MISC, 7), 1);                // BFULL
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < TC_NROWC; i += blockDim.x) sh.sRow[i] = tc.rowc[(size_t)r * TC_NROWC + i];
    for (int i = threadIdx.x; i < TC_NOUT + 4; i += blockDim.x) sh.sCst[i] = tc.cstb[(size_t)r * (TC_NOUT + 4) + i];
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const int my_iters = slot < nslots ? (n_mtiles - slot + nslots - 1) / nslots : 0;
    const int nslab = my_iters * nreg;                          // 16 KB slabs this CTA streams

    if (warp == 0) {
        // ===================================================================== TMA producer
        if (lane == 0 && my_iters > 0) {
            mbar_expect_tx(tc_bar(bar0, TCB_MISC, 7), (uint32_t)tc_b_bytes(nreg));
            for (int rg = 0; rg < nreg; rg++)
                tma_load_2d(smem_u32(sB + (size_t)rg * TC_NPAD * 128), &map_b, rg * 128, r * TC_NPAD, tc_bar(bar0, TCB_MISC, 7));
            int s = 0, ph = 0;
            for (int it = 0; it < my_iters; it++) {
                const int mt = slot + it * nslots;
                for (int rg = 0; rg < nreg; rg++) {
                    mbar_wait_sleep(tc_bar(bar0, TCB_A_FREE, s), ph ^ 1);
                    if (rg == 0) TC_DBG(sc, it, 0);
                    mbar_expect_tx(tc_bar(bar0, TCB_FULL_A, s), TC_REGION_BYTES);
                    tma_load_2d_hint(smem_u32(sA + (size_t)s * TC_REGION_BYTES), &map_a, rg * 128, mt * 128, tc_bar(bar0, TCB_FULL_A, s),
                                     TC_L2_EVICT_FIRST);
                    if (++s == nstage) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================================== MMA issuer
        if (lane == 0 && my_iters > 0) {
            mbar_wait_sleep(tc_bar(bar0, TCB_MISC, 7), 0);
            int s = 0, ph = 0;
            for (int it = 0; it < my_iters; it++) {
                const int ts = it & 1, u = it >> 1;              // TMEM stage
                const uint32_t d = tmem_base + (uint32_t)(ts * 256);
                for (int rg = 0; rg < nreg; rg++) {
                    mbar_wait_sleep(tc_bar(bar0, TCB_XORED, s), ph);
                    if (rg == 0) mbar_wait(tc_bar(bar0, TCB_MISC, 2 + ts), (u & 1) ^ 1);
                    tc_fence_after();
                    if (rg == 0) TC_DBG(sc, it, 3);
                    const uint32_t a0 = smem_u32(sA + (size_t)s * TC_REGION_BYTES);
                    const uint32_t b0 = smem_u32(sB + (size_t)rg * TC_NPAD * 128);
#pragma unroll
                    for (int ks = 0; ks < 4; ks++)
                        umma_i8(d, umma_desc(a0 + ks * 32), umma_desc(b0 + ks * 32), tc.idesc, (rg | ks) ? 1u : 0u);
                    umma_commit(tc_bar(bar0, TCB_A_FREE, s));    // the staged bytes are dead once the MMAs retire
                    if (++s == nstage) { s = 0; ph ^= 1; }
                }
                umma_commit(tc_bar(bar0, TCB_MISC, 4 + it % TC_EPI_GROUPS));
                TC_DBG(sc, it, 4);
            }
        }
    } else if (warp < 4) {
        // ===================================================================== sign fix-up
        const int tx = threadIdx.x - 64;
        const uint32_t m = tc.xor_word;
        int s = 0, ph = 0;
        for (int k = 0; k < nslab; k++) {
            mbar_wait_sleep(tc_bar(bar0, TCB_FULL_A, s), ph);
            if (threadIdx.x == 64 && (k % nreg) == 0) TC_DBG(sc, k / nreg, 1);
            if (m) {
                uint4 *base = reinterpret_cast<uint4 *>(sA + (size_t)s * TC_REGION_BYTES) + tx;
                uint4 v[16];
#pragma unroll
                for (int i = 0; i < 16; i++) v[i] = base[i * 64];
#pragma unroll
                for (int i = 0; i < 16; i++) {
                    v[i].x ^= m; v[i].y ^= m; v[i].z ^= m; v[i].w ^= m;
                    base[i * 64] = v[i];
                }
                fence_proxy_async();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(tc_bar(bar0, TCB_XORED, s));
            if (threadIdx.x == 64 && (k % nreg) == nreg - 1) TC_DBG(sc, k / nreg, 2);
            if (++s == nstage) { s = 0; ph ^= 1; }
        }
    } else {
        // ===================================================================== epilogue
        tc_epilogue<IQ>(pl, tc, sc, sh, tmem_base, warp - 4, lane, r, slot, nslots, my_iters, total_wtiles);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
    }
}
