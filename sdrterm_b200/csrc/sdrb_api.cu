// sdrb_api.cu -- C ABI of libsdrterm_b200.so (see include/sdrterm_b200.h).
// Host side: table upload, scratch, kernel launch sequence, double-buffered host streaming.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <mutex>
#include <type_traits>
#include <vector>

#include "../../include/sdrterm_b200.h"
#include "sdrb_kernels.cuh"
#include "sdrb_tc.cuh"
#include "sdrb_finish.cuh"
#include "sdrb_spectrum.cuh"
#include "sdrb_seamless.cuh"

namespace {

thread_local std::string g_error;

struct Slot {
    uint8_t *raw = nullptr;   // device staging for host-path input
    double *out = nullptr;    // device staging for host-path output
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    double *host_out = nullptr;
    size_t nchunks = 0;
};

}  // namespace

struct sdrb_handle {
    sdrb_config cfg{};
    DevPlan pl{};
    Scratch sc{};
    std::vector<void *> owned;      // device allocations to free
    Slot slot[2];
    cudaEvent_t iq_done = nullptr;  // orders the IQ-state chain between slots
    size_t max_chunks = 0;
    int enc_code = 0;
    int tpc = 1, warps = 4;
    size_t main_smem = 0, demod_smem = 0;
    bool finish_on = false;         // fused k_finish instead of k_fixup + k_demod
    size_t finish_smem = 0;
    int keep_y = 0;
    long long launches = 0;
    size_t last_nchunks = 0;
    bool profiling = false;
    cudaEvent_t pev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    bool pev_valid[5] = {false, false, false, false, false};
    std::string error;
    // tensor-core block front end (k_tc)
    bool tc_on = false;
    TcDev tc{};
    CUtensorMap map_b{};
    size_t tc_smem = 0;
    int num_sms = 148;
    int reserved_sms = 0;           // SMs the persistent kernels leave free (for a collective running beside them)
    double2 *x0_buf = nullptr;      // sdrb_keep_x0
    int smooth_w = 0, smooth_nhead = 0, smooth_ntail = 0, smooth_lo = 0;   // --smooth-output (window 0 = off)
    double *smooth_S = nullptr, *smooth_tmp = nullptr;
    // seamless streaming (cfg.seamless): window of unemitted chunks in slots 0..nwin-1 of the scratch
    bool seamless = false;
    SeamDev sd{};
    long long seen = 0, emitted = 0;   // chunks of the current stream taken in / emitted
    int nwin = 0;
};

namespace {

int fail(sdrb_handle *h, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->error = buf;
    g_error = buf;
    return code;
}

#define CK(h, call)                                                                        \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess)                                                             \
            return fail(h, SDRB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                               \
    } while (0)

int enc_code_of(char c)
{
    switch (c) {
    case 'b': return ENC_b; case 'B': return ENC_B; case 'h': return ENC_h; case 'H': return ENC_H;
    case 'i': return ENC_i; case 'I': return ENC_I; case 'f': return ENC_f; case 'd': return ENC_d;
    case 'Z': return ENC_Z; default: return -1;
    }
}
int itemsize_of(int code)
{
    static const int sz[] = {1, 1, 2, 2, 4, 4, 4, 8, 8};
    return sz[code];
}

// The one place a runtime encoding code becomes a kernel template argument: calls
// f(std::integral_constant<int, ENC_x>{}) and returns its result.
template <class F>
int with_enc(sdrb_handle *h, int code, F &&f)
{
    switch (code) {
    case ENC_b: return f(std::integral_constant<int, ENC_b>{});
    case ENC_B: return f(std::integral_constant<int, ENC_B>{});
    case ENC_h: return f(std::integral_constant<int, ENC_h>{});
    case ENC_H: return f(std::integral_constant<int, ENC_H>{});
    case ENC_i: return f(std::integral_constant<int, ENC_i>{});
    case ENC_I: return f(std::integral_constant<int, ENC_I>{});
    case ENC_f: return f(std::integral_constant<int, ENC_f>{});
    case ENC_d: return f(std::integral_constant<int, ENC_d>{});
    case ENC_Z: return f(std::integral_constant<int, ENC_Z>{});
    }
    return fail(h, SDRB_ERR_ARG, "bad encoding code %d", code);
}

template <typename T>
int upload(sdrb_handle *h, const T *src, size_t count, const T **dst)
{
    void *d = nullptr;
    if (count == 0) count = 1;
    CK(h, cudaMalloc(&d, count * sizeof(T)));
    h->owned.push_back(d);
    if (src) CK(h, cudaMemcpy(d, src, count * sizeof(T), cudaMemcpyHostToDevice));
    else CK(h, cudaMemset(d, 0, count * sizeof(T)));
    *dst = static_cast<const T *>(d);
    return 0;
}
template <typename T>
int dalloc(sdrb_handle *h, size_t count, T **dst)
{
    void *d = nullptr;
    if (count == 0) count = 1;
    CK(h, cudaMalloc(&d, count * sizeof(T)));
    h->owned.push_back(d);
    *dst = static_cast<T *>(d);
    return 0;
}

inline double2 c2(const double *a, size_t i) { return make_double2(a[2 * i], a[2 * i + 1]); }
inline double2 hmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }
bool is_ssb(int demod) { return demod == SDRB_USB || demod == SDRB_LSB; }
// the finish-kernel instance of a demodulation (OUT_REAL / OUT_IQ / OUT_SSB)
int out_kind(int demod) { return demod == SDRB_IQ ? OUT_IQ : (is_ssb(demod) ? OUT_SSB : OUT_REAL); }

std::vector<double2> make_twiddles(int n)
{
    std::vector<double2> tw(n > 0 ? n : 1);
    const long double two_pi = 6.283185307179586476925286766559005768L;
    for (int k = 0; k < n; k++) {
        long double a = -two_pi * (long double)k / (long double)n;
        tw[k] = make_double2((double)cosl(a), (double)sinl(a));
    }
    return tw;
}

int env_int(const char *name, int dflt);
int launch_tc(sdrb_handle *h, const uint8_t *raw, size_t nch, cudaStream_t st, bool iq);

enum { PH_MAIN = 1, PH_IQSCAN = 2, PH_FINISH = 4, PH_ALL = 7 };

// ------------------------------------------------------------------ tensor-core front end
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
encode_tiled_fn get_encode_tiled()
{
    static encode_tiled_fn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<encode_tiled_fn>(p);
    }
    return fn;
}

// 2-D byte tensor [rows][K] (row pitch K), box = 128 bytes x box_rows, 128B swizzle.
int make_byte_map(sdrb_handle *h, CUtensorMap *map, const void *base, uint64_t rows, uint32_t K, uint32_t box_rows)
{
    encode_tiled_fn enc = get_encode_tiled();
    if (!enc) return fail(h, SDRB_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
    cuuint64_t dims[2] = {K, rows};
    cuuint64_t strides[1] = {K};
    cuuint32_t box[2] = {128, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, SDRB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return 0;
}

template <bool IQ>
int launch_tc_t(sdrb_handle *h, const CUtensorMap &map_a, int n_mtiles, int total_wtiles, cudaStream_t st)
{
    // one row of the bank per CTA: the grid is a whole number of row groups
    const int R = h->pl.R;
    const int slots = std::max(1, std::min((h->num_sms - h->reserved_sms) / R, n_mtiles));
    k_tc<IQ><<<slots * R, TC_THREADS, h->tc_smem, st>>>(h->pl, h->tc, h->sc, map_a, h->map_b, n_mtiles, total_wtiles);
    return 0;
}

int launch_tc(sdrb_handle *h, const uint8_t *raw, size_t nch, cudaStream_t st, bool iq)
{
    // GEMM rows are super-blocks of two blocks: [nch * Mf / 2][K] bytes, 128 rows per MMA tile
    const uint64_t rows = (uint64_t)nch * h->pl.Mf / 2;
    CUtensorMap map_a;
    int rc = make_byte_map(h, &map_a, raw, rows, (uint32_t)h->tc.K, 128);
    if (rc) return rc;
    const int n_mtiles = (int)((rows + 127) / 128);
    const int total_wtiles = (int)(rows / 32);
    return iq ? launch_tc_t<true>(h, map_a, n_mtiles, total_wtiles, st) : launch_tc_t<false>(h, map_a, n_mtiles, total_wtiles, st);
}

template <bool IQ>
int tc_attr(sdrb_handle *h)
{
    CK(h, cudaFuncSetAttribute(k_tc<IQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->tc_smem));
    return 0;
}

int setup_tc(sdrb_handle *h, const sdrb_tables *tab)
{
    if (!tab->tc_enable) return 0;
    const int R = h->pl.R;
    if ((tab->tc_K != 256 && tab->tc_K != 512) || tab->tc_nout != TC_NOUT || tab->tc_ncol != TC_NCOL ||
        tab->tc_isz < 1 || tab->tc_isz > 2 || tab->tc_npad != TC_NPAD || tab->tc_nrowc != TC_NROWC ||
        tab->tc_K != 2 * h->pl.q * h->pl.sb || h->pl.rem != 0 || h->pl.cnt_last != SDRB_TB || (h->pl.Mf / 2) % 128 ||
        h->pl.q < h->pl.edge + 1 || h->pl.normalize || !tab->tc_Bq || !tab->tc_cst || !tab->tc_rowc)
        return fail(h, SDRB_ERR_ARG, "tensor-core tables do not match the configuration");
    cudaDeviceProp prop;
    CK(h, cudaGetDeviceProperties(&prop, h->cfg.device));
    h->num_sms = prop.multiProcessorCount;
    if (R > TC_MAX_R) return 0;              // wider banks take the FP64 block kernel
    TcDev &tc = h->tc;
    tc.K = tab->tc_K; tc.isz = tab->tc_isz;
    tc.nregion = tc.K / 128;
    memcpy(&tc.xor_word, tab->tc_xor, 4);
    for (int i = 0; i < 16; i++)
        if (tab->tc_xor[i] != tab->tc_xor[i & 3]) return fail(h, SDRB_ERR_ARG, "XOR pattern is not 4-periodic");
    // instruction descriptor: D = s32, A = s8 / u8 (tc_a_signed), B = s8, N, M
    tc.idesc = (2u << 4) | ((tab->tc_a_signed ? 1u : 0u) << 7) | (1u << 10) | ((uint32_t)(TC_NPAD >> 3) << 17) | ((128u >> 4) << 24);
    tc.scale = ldexp(1.0, -tab->tc_S);
    tc.scale16 = ldexp(1.0, 16 - tab->tc_S);
    tc.scale_yl = ldexp(1.0, -tab->tc_S_yl);
    tc.scale16_yl = ldexp(1.0, 16 - tab->tc_S_yl);
    int rc = upload(h, reinterpret_cast<const double2 *>(tab->tc_rowc), (size_t)R * TC_NROWC, &tc.rowc);
    if (rc) return rc;
    std::vector<double> cstb((size_t)R * (TC_NOUT + 4));
    for (int r = 0; r < R; r++)
        for (int o = 0; o < TC_NOUT + 4; o++) {
            const double sc = o < 36 ? tc.scale : (o < TC_NOUT ? tc.scale_yl : 1.0);
            cstb[(size_t)r * (TC_NOUT + 4) + o] = tab->tc_cst[(size_t)r * (TC_NOUT + 4) + o] - TC_BIAS32 * sc;
        }
    rc = upload(h, cstb.data(), cstb.size(), &tc.cstb);
    if (rc) return rc;
    const int8_t *d_bq = nullptr;
    rc = upload(h, tab->tc_Bq, (size_t)R * TC_NPAD * tc.K, &d_bq);
    if (rc) return rc;
    rc = make_byte_map(h, &h->map_b, d_bq, (uint64_t)R * TC_NPAD, (uint32_t)tc.K, (uint32_t)TC_NPAD);
    if (rc) return rc;
    // the A ring takes whatever shared memory the B slice leaves (227 KB per CTA on sm_100)
    const size_t cap = 227 * 1024;
    const size_t fixed = tc_fixed_bytes(tc.nregion);
    int nstage = fixed < cap ? (int)((cap - fixed) / TC_REGION_BYTES) : 0;
    nstage = std::min(nstage, env_int("SDRB_TC_ASTAGES", TC_MAX_ASTAGES));
    nstage = std::min(nstage, TC_MAX_ASTAGES);
    if (nstage < 2) return fail(h, SDRB_ERR_ARG, "k_tc: no room for the A ring (%zu bytes fixed)", fixed);
    tc.nstage = nstage;
    h->tc_smem = tc_smem_bytes(tc.nregion, nstage);
    if ((rc = tc_attr<true>(h)) || (rc = tc_attr<false>(h))) return rc;
    h->tc_on = true;
    return 0;
}

template <int ENC, bool IQ>
int launch_chain_t(sdrb_handle *h, const uint8_t *raw, size_t nch, double *out, cudaStream_t st, int phases)
{
    const DevPlan &pl = h->pl;
    const bool prof = h->profiling && phases == PH_ALL;
    auto mark = [&](int i) {
        if (prof) { cudaEventRecord(h->pev[i], st); h->pev_valid[i] = true; }
    };
    if (prof) for (int i = 0; i < 5; i++) h->pev_valid[i] = false;
    mark(0);
    if (phases & PH_MAIN) {
        if (h->tc_on && ((uintptr_t)raw & 15) == 0) {
            int rc = launch_tc(h, raw, nch, st, IQ);
            if (rc) return rc;
        } else {
            const int groups = (pl.ntiles + h->tpc - 1) / h->tpc;
            k_main<ENC, IQ><<<(unsigned)(nch * groups), 32 * h->warps, h->main_smem, st>>>(pl, h->sc, raw, (int)nch, h->tpc);
        }
        h->launches++;
    }
    mark(1);
    if ((phases & PH_IQSCAN) && IQ) {
        // chunk gains -> the chunk scan (offset at every chunk start) -> the offsets at the tile
        // starts, which k_finish derives itself
        const bool finish_tiles = h->finish_on && pl.ntiles <= 32 && !h->seamless;
        const unsigned gw = (unsigned)((nch + 7) / 8);    // warp <-> chunk, 8 warps per CTA
        k_iqgain<ENC><<<gw, 256, 0, st>>>(pl, h->sc, raw, (int)nch);
        k_iqscan_c<<<1, 1024, 0, st>>>(pl, h->sc, (int)nch);
        if (!finish_tiles) k_iqtiles<<<gw, 256, 0, st>>>(pl, h->sc, (int)nch);
        h->launches += finish_tiles ? 2 : 3;
    }
    mark(2);
    if ((phases & PH_FINISH) && h->finish_on) {
        const size_t items = nch * (size_t)pl.R;
        const unsigned grid = (unsigned)std::min<size_t>((items + FIN_WARPS - 1) / FIN_WARPS, (size_t)(h->num_sms - h->reserved_sms) * 2);
        if (pl.demod == SDRB_IQ)
            k_finish<ENC, OUT_IQ><<<grid, 32 * FIN_WARPS, h->finish_smem, st>>>(pl, h->sc, raw, out, (int)nch, h->keep_y);
        else if (is_ssb(pl.demod))
            k_finish<ENC, OUT_SSB><<<grid, 32 * FIN_WARPS, h->finish_smem, st>>>(pl, h->sc, raw, out, (int)nch, h->keep_y);
        else
            k_finish<ENC, OUT_REAL><<<grid, 32 * FIN_WARPS, h->finish_smem, st>>>(pl, h->sc, raw, out, (int)nch, h->keep_y);
        h->launches++;
        mark(3);
        mark(4);
    } else if (phases & PH_FINISH) {
        k_fixup<ENC><<<(unsigned)(nch * pl.R), 128, 0, st>>>(pl, h->sc, raw, (int)nch);
        h->launches++;
        mark(3);
        if (pl.demod == SDRB_IQ)
            k_demod<OUT_IQ><<<(unsigned)(nch * pl.R), 128, 0, st>>>(pl, h->sc.y, out, nullptr, nullptr, (int)nch, pl.demod, 0,
                                                                    pl.be_out);
        else if (is_ssb(pl.demod))
            k_demod<OUT_SSB><<<(unsigned)(nch * pl.R), 128, h->demod_smem, st>>>(pl, h->sc.y, out, h->sc.fftbuf, h->sc.zrow,
                                                                                 (int)nch, pl.demod, 1, pl.be_out);
        else
            k_demod<OUT_REAL><<<(unsigned)(nch * pl.R), 128, h->demod_smem, st>>>(pl, h->sc.y, out, h->sc.fftbuf, h->sc.zrow,
                                                                                  (int)nch, pl.demod, 1, pl.be_out);
        h->launches++;
        mark(4);
    }
    if ((phases & PH_FINISH) && h->smooth_w > 0 && !pl.be_out) {
        const size_t nseg = nch * (size_t)pl.R, bytes = nseg * pl.M * sizeof(double);
        k_savgol<<<(unsigned)std::min<size_t>(nseg, (size_t)h->num_sms * 8), 256, 0, st>>>(out, h->smooth_tmp, h->smooth_S,
                                                                                        h->smooth_w, h->smooth_nhead, h->smooth_ntail, h->smooth_lo, pl.M, nseg);
        CK(h, cudaMemcpyAsync(out, h->smooth_tmp, bytes, cudaMemcpyDeviceToDevice, st));
        h->launches++;
    }
    CK(h, cudaGetLastError());
    return 0;
}

int launch_chain(sdrb_handle *h, const uint8_t *raw, size_t nch, double *out, cudaStream_t st, int phases = PH_ALL)
{
    if ((phases & PH_FINISH) && h->pl.demod == SDRB_IQ && ((uintptr_t)out & 15))
        return fail(h, SDRB_ERR_ARG, "iq output is stored as 16-byte (Re, Im) pairs: `out` must be 16-byte aligned");
    return with_enc(h, h->enc_code, [&](auto enc) {
        constexpr int E = decltype(enc)::value;
        return h->pl.correct_iq ? launch_chain_t<E, true>(h, raw, nch, out, st, phases)
                                : launch_chain_t<E, false>(h, raw, nch, out, st, phases);
    });
}

template <int ENC, bool IQ>
int set_smem_attr_t(sdrb_handle *h)
{
    CK(h, cudaFuncSetAttribute(k_main<ENC, IQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->main_smem));
    if (h->finish_on) {
        const int ok = out_kind(h->pl.demod);
        CK(h, cudaFuncSetAttribute(ok == OUT_IQ ? k_finish<ENC, OUT_IQ> : (ok == OUT_SSB ? k_finish<ENC, OUT_SSB> : k_finish<ENC, OUT_REAL>),
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->finish_smem));
    }
    return 0;
}
int set_smem_attr(sdrb_handle *h)
{
    return with_enc(h, h->enc_code, [&](auto enc) {
        constexpr int E = decltype(enc)::value;
        return h->pl.correct_iq ? set_smem_attr_t<E, true>(h) : set_smem_attr_t<E, false>(h);
    });
}

int env_int(const char *name, int dflt)
{
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

}  // namespace

extern "C" {

const char *sdrb_global_error(void) { return g_error.c_str(); }
const char *sdrb_last_error(const sdrb_handle *h) { return h ? h->error.c_str() : g_error.c_str(); }

int sdrb_create(const sdrb_config *cfg, const sdrb_tables *tab, sdrb_handle **out)
{
    if (!cfg || !tab || !out) return fail(nullptr, SDRB_ERR_ARG, "null argument");
    if (cfg->abi_version != SDRB_ABI_VERSION) return fail(nullptr, SDRB_ERR_ARG, "ABI version mismatch");
    const int code = enc_code_of(cfg->enc);
    if (code < 0) return fail(nullptr, SDRB_ERR_ARG, "unknown encoding '%c'", cfg->enc);
    if (cfg->q < 2 || cfg->q > SDRB_MAX_DECIMATION)
        return fail(nullptr, SDRB_ERR_ARG, "decimation %d outside 2..%d", cfg->q, SDRB_MAX_DECIMATION);
    if (cfg->R < 1 || cfg->edge < 1 || cfg->N <= cfg->edge + 1 || cfg->max_chunks < 1 || cfg->n_out_sections < 0 ||
        cfg->n_out_sections > 4)
        return fail(nullptr, SDRB_ERR_ARG, "bad geometry");
    {   // k_fixup stages (edge+1) head samples and nend = max(rem, edge+1) window samples in shared memory
        const int rem = cfg->N % cfg->q;
        if (cfg->edge + 1 + std::max(rem, cfg->edge + 1) > SDRB_NEDGE)
            return fail(nullptr, SDRB_ERR_ARG, "filter pad %d too long for the fix-up kernel", cfg->edge);
    }
    {
        const void *need[] = {tab->p, tab->P, tab->rho, tab->rho_p, tab->c, tab->zhat, tab->xi, tab->Ec, tab->Oc,
                              tab->Ppow, tab->pk, tab->Pt, tab->bx, tab->bnd, tab->lam_j, tab->lam_k, tab->mu_k,
                              tab->T2, tab->T3, tab->T1, tab->Ehead, tab->Eend, tab->alpha, tab->alphaT, tab->beta,
                              tab->betaT, tab->gamma, tab->phE, tab->psiY, tab->use_nco};
        for (const void *ptr : need)
            if (!ptr) return fail(nullptr, SDRB_ERR_ARG, "a required table pointer is NULL");
        if (cfg->n_out_sections > 0 && !tab->out_sos) return fail(nullptr, SDRB_ERR_ARG, "out_sos is NULL");
    }
    if (cfg->N / cfg->q < 1) return fail(nullptr, SDRB_ERR_ARG, "chunk shorter than one block");
    if (cfg->demod > SDRB_LSB) return fail(nullptr, SDRB_ERR_ARG, "unknown demodulation %d", (int)cfg->demod);
    if (cfg->demod == SDRB_IQ && cfg->n_out_sections != 0)
        return fail(nullptr, SDRB_ERR_ARG, "iq output has no output low-pass (n_out_sections must be 0)");
    if (is_ssb(cfg->demod)) {
        // the band-pass is the rotated prototype: sections, a rotation inside (0, pi/2) of the
        // sideband's sign, and the table of its powers that matches it
        const double om = tab->ssb_omega, sgn = cfg->demod == SDRB_USB ? 1.0 : -1.0;
        if (cfg->n_out_sections < 1 || !tab->out_sos || !tab->ssb_rot || !(sgn * om > 0.0) || !(sgn * om < M_PI / 2))
            return fail(nullptr, SDRB_ERR_ARG, "usb/lsb needs the prototype sections and a rotation 0 < %s < pi/2 (got %g)",
                        cfg->demod == SDRB_USB ? "Omega" : "-Omega", om);
        if (std::fabs(tab->ssb_rot[0] - 1.0) > 1e-12 || std::fabs(tab->ssb_rot[1]) > 1e-12 ||
            std::fabs(tab->ssb_rot[2] - std::cos(om)) > 1e-12 || std::fabs(tab->ssb_rot[3] - std::sin(om)) > 1e-12)
            return fail(nullptr, SDRB_ERR_ARG, "ssb_rot does not start 1, e^{j Omega}");
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, SDRB_ERR_CUDA, "no CUDA device: libsdrterm_b200 has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, SDRB_ERR_ARG, "bad device ordinal");

    sdrb_handle *h = new sdrb_handle();
    h->cfg = *cfg;
    h->enc_code = code;
    h->max_chunks = (size_t)cfg->max_chunks;
    int rc = 0;
    auto bail = [&](int c) { std::string e = h->error; sdrb_destroy(h); g_error = e; return c; };
    if (cudaSetDevice(cfg->device) != cudaSuccess) return bail(fail(h, SDRB_ERR_CUDA, "cudaSetDevice failed"));

    DevPlan &pl = h->pl;
    pl.enc = code; pl.itemsize = itemsize_of(code); pl.swap = cfg->swap; pl.correct_iq = cfg->correct_iq;
    pl.normalize = cfg->normalize; pl.demod = cfg->demod; pl.be_out = cfg->big_endian_out;
    pl.q = cfg->q; pl.N = cfg->N; pl.edge = cfg->edge; pl.L = cfg->N + 2 * cfg->edge;
    pl.Mf = cfg->N / cfg->q; pl.rem = cfg->N - pl.Mf * cfg->q; pl.M = pl.Mf + (pl.rem ? 1 : 0);
    pl.W = cfg->demod == SDRB_IQ ? 2 * pl.M : pl.M;
    pl.ssb_omega = is_ssb(cfg->demod) ? tab->ssb_omega : 0.0;
    pl.ntiles = (pl.Mf + SDRB_TB - 1) / SDRB_TB; pl.cnt_last = pl.Mf - (pl.ntiles - 1) * SDRB_TB;
    pl.Hq = (cfg->q + 1) / 2; pl.KS = (pl.Hq + 3) / 4; pl.R = cfg->R;
    pl.RL = tab->RL;
    if (pl.RL != pl.KS) return bail(fail(h, SDRB_ERR_ARG, "RL %d does not match ceil(Hq/4) = %d", pl.RL, pl.KS));
    pl.sb = 2 * pl.itemsize;
    for (int i = 0; i < 8; i++) { pl.run_len[i] = tab->run_len[i]; pl.lam_run[i] = tab->lam_run[i]; }
    pl.lam_inv = tab->lam_inv;
    pl.sos_ns = 2 * cfg->n_out_sections; pl.sos_Lseg = tab->sos_Lseg;
    if (cfg->n_out_sections > 0) {
        if (!tab->sos_CA || !tab->sos_AP || tab->sos_Lseg * 32 < pl.M)
            return bail(fail(h, SDRB_ERR_ARG, "output SOS segment tables missing or too short"));
        for (int i = 0; i < 5 * pl.sos_ns * pl.sos_ns; i++) pl.sos_AP[i] = tab->sos_AP[i];
    }
    pl.ws = std::min(pl.q * pl.Mf, pl.N - 1 - pl.edge); pl.nend = pl.N - pl.ws;
    pl.k_bnd = tab->k_bnd; pl.nsec_out = cfg->n_out_sections;
    pl.Liq = cfg->correct_iq ? cfg->iq_L : 0.0; pl.lam = tab->lam; pl.lam_q = tab->lam_q; pl.lam_N = tab->lam_N;
    pl.g0 = tab->g0; pl.d = tab->d; pl.norm_xmin = cfg->norm_xmin; pl.norm_k = cfg->norm_k;
    pl.lam_tile[0] = tab->lam_tile[0]; pl.lam_tile[1] = tab->lam_tile[1];
    {
        double v = tab->lam_q;
        for (int i = 0; i < 5; i++) { pl.lamq_pow[i] = v; v *= v; }
    }
    for (int i = 0; i < SDRB_NP; i++) {
        pl.p[i] = c2(tab->p, i); pl.P[i] = c2(tab->P, i); pl.rho[i] = c2(tab->rho, i);
        pl.rho_p[i] = c2(tab->rho_p, i); pl.c[i] = c2(tab->c, i); pl.zhat[i] = c2(tab->zhat, i);
    }
    for (int i = 0; i < SDRB_NP * SDRB_NP; i++) pl.xi[i] = c2(tab->xi, i);
    for (int i = 0; i < 6 * cfg->n_out_sections; i++) pl.out_sos[i] = tab->out_sos[i];

    const int q = pl.q, R = pl.R, Hq = pl.Hq, KS = pl.KS, nt = pl.ntiles, M = pl.M;
    // DMMA A fragments: lane -> (row o = lane>>2: mode o>>1, Re/Im o&1 ; col k = lane&3)
    std::vector<double> afrag((size_t)KS * 2 * 32, 0.0);
    for (int s = 0; s < KS; s++)
        for (int lane = 0; lane < 32; lane++) {
            const int o = lane >> 2, k = lane & 3, j = k * KS + s, m = o >> 1, e = o & 1;
            if (j < Hq && j < (k + 1) * KS) {
                afrag[((size_t)2 * s) * 32 + lane] = tab->Ec[2 * ((size_t)m * Hq + j) + e];
                afrag[((size_t)2 * s + 1) * 32 + lane] = tab->Oc[2 * ((size_t)m * Hq + j) + e];
            }
        }
    std::vector<double2> rw((size_t)(SDRB_TB + 1) * 8), rt((size_t)(SDRB_TB + 1) * 8);
    for (int l = 0; l <= SDRB_TB; l++)
        for (int i = 0; i < 8; i++) {
            const double2 pp = c2(tab->Ppow, (size_t)l * 8 + i);
            rw[(size_t)l * 8 + i] = hmul(pl.rho[i], pp);
            rt[(size_t)l * 8 + i] = hmul(pl.rho_p[i], pp);
        }
    std::vector<double2> prot((size_t)R * 16);
    for (int r = 0; r < R; r++) {
        const double2 eps = c2(tab->T3, (size_t)r * (SDRB_TB + 1) + 1);
        for (int i = 0; i < 8; i++) {
            prot[(size_t)r * 16 + i] = hmul(make_double2(eps.x, -eps.y), pl.P[i]);
            prot[(size_t)r * 16 + 8 + i] = hmul(eps, pl.P[i]);
        }
    }
    const int h2 = M >> 1;
    pl.fft_ok = (M == 2 * h2) && is_pow2(h2) ? 1 : 0;
    pl.fft_n = pl.fft_ok ? M : 0;
    if (cfg->demod == SDRB_FM && !pl.fft_ok && !tab->fm_interp)
        return bail(fail(h, SDRB_ERR_ARG, "FM with M=%d needs the dense interpolation table", M));
    std::vector<double2> tw = make_twiddles(pl.fft_n);

#define UP(expr) do { rc = (expr); if (rc) return bail(rc); } while (0)
    UP(upload(h, afrag.data(), afrag.size(), &pl.Afrag));
    UP(upload(h, tab->lam_j, (size_t)q + 1, &pl.lam_j));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->Ppow), (size_t)(SDRB_TB + 1) * 8, &pl.Ppow));
    if (!tab->pk || !tab->lam_k || !tab->mu_k || !tab->Pt || !tab->bx) return bail(fail(h, SDRB_ERR_ARG, "pole / IQ power tables missing"));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->pk), (size_t)(pl.edge + 1) * 8, &pl.pk));
    for (int i = 0; i < 33; i++) { pl.lam_pw[i] = tab->lam_k[i]; pl.mu_pw[i] = tab->mu_k[i]; }
    UP(upload(h, reinterpret_cast<const double2 *>(tab->Pt), (size_t)nt * 8, &pl.Pt));
    for (int i = 0; i < SDRB_NP; i++) pl.bx[i] = c2(tab->bx, i);
    UP(upload(h, rw.data(), rw.size(), &pl.RW));
    UP(upload(h, rt.data(), rt.size(), &pl.RT));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->bnd), (size_t)M * 8, &pl.bnd));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->T2), (size_t)R * q, &pl.T2));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->T3), (size_t)R * (SDRB_TB + 1), &pl.T3));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->T1), (size_t)R * nt, &pl.T1));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->Ehead), (size_t)R * (pl.edge + 1), &pl.Ehead));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->Eend), (size_t)R * pl.nend, &pl.Eend));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->alpha), (size_t)R * 8, &pl.alpha));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->alphaT), (size_t)R * 8, &pl.alphaT));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->beta), (size_t)R * 8, &pl.beta));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->betaT), (size_t)R * 8, &pl.betaT));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->gamma), (size_t)R, &pl.gamma));
    UP(upload(h, reinterpret_cast<const double2 *>(tab->phE), (size_t)R, &pl.phE));
    {   // reciprocals and output weights derived from them (host doubles; |beta - 1| << 1)
        std::vector<double2> binv((size_t)R * 8), binvT((size_t)R * 8), rb((size_t)R * 8), rbT((size_t)R * 8);
        auto hinv = [](double2 a) { const double d = a.x * a.x + a.y * a.y; return make_double2(a.x / d, -a.y / d); };
        for (int r = 0; r < R; r++)
            for (int i = 0; i < 8; i++) {
                const double2 b = c2(tab->beta, (size_t)r * 8 + i), bT = c2(tab->betaT, (size_t)r * 8 + i);
                binv[(size_t)r * 8 + i] = hinv(b); binvT[(size_t)r * 8 + i] = hinv(bT);
                rb[(size_t)r * 8 + i] = hmul(pl.rho[i], b); rbT[(size_t)r * 8 + i] = hmul(pl.rho_p[i], bT);
            }
        UP(upload(h, binv.data(), binv.size(), &pl.binv));
        UP(upload(h, binvT.data(), binvT.size(), &pl.binvT));
        UP(upload(h, rb.data(), rb.size(), &pl.rb));
        UP(upload(h, rbT.data(), rbT.size(), &pl.rbT));
    }
    UP(upload(h, reinterpret_cast<const double2 *>(tab->psiY), (size_t)2 * R * SDRB_TB, &pl.psiY));
    UP(upload(h, prot.data(), prot.size(), &pl.Prot));
    UP(upload(h, tw.data(), tw.size(), &pl.tw));
    UP(upload(h, tab->use_nco, (size_t)R, &pl.use_nco));
    pl.sos_CA = nullptr;
    if (cfg->n_out_sections > 0) UP(upload(h, tab->sos_CA, (size_t)pl.sos_Lseg * pl.sos_ns, &pl.sos_CA));
    pl.fm_interp = nullptr;
    if (cfg->demod == SDRB_FM && !pl.fft_ok) UP(upload(h, tab->fm_interp, (size_t)M * h2, &pl.fm_interp));
    pl.ssb_rot = nullptr;
    if (is_ssb(cfg->demod)) UP(upload(h, reinterpret_cast<const double2 *>(tab->ssb_rot), (size_t)M + 1, &pl.ssb_rot));

    // launch geometry
    auto smem_for = [&](int tpc, int w) {
        return (size_t)tpc * main_tile_bytes(pl.RL, pl.sb) + (size_t)w * main_warp_bytes();
    };
    // k_main: a CTA's warps share TPC staged tiles and take (tile, row) items in rounds
    // (more than one tile per CTA measured slower for banks: 33 rows, TPC 1/2/3 -> 205/191/153 G)
    const int tpc_auto = R == 1 ? 2 : 1;
    // warps per CTA for a bank: 8 (two CTAs of 126 registers per SM).  Measured, float32 q = 64,
    // G VFO*samples/s at 257/65/33 rows: W=8 326/308/290, W=7 306/290/286, W=6 303/291/277,
    // W=5 311/304/292 (microbench/bank_rows.py).
    const int warps_auto = R == 1 ? 2 : (R >= 8 ? 8 : 4);
    h->tpc = env_int("SDRB_TPC", tpc_auto);
    if (h->tpc > pl.ntiles) h->tpc = pl.ntiles;
    h->warps = env_int("SDRB_WARPS", R == 1 ? h->tpc : warps_auto);
    if (h->tpc < 1) h->tpc = 1;
    if (h->warps < 1) h->warps = 1;
    if (h->warps > 8) h->warps = 8;
    while (h->tpc > 1 && smem_for(h->tpc, h->warps) > 220 * 1024) h->tpc--;
    while (h->warps > 1 && smem_for(h->tpc, h->warps) > 220 * 1024) h->warps--;
    h->main_smem = smem_for(h->tpc, h->warps);
    if (h->main_smem > 227 * 1024) return bail(fail(h, SDRB_ERR_ARG, "decimation %d needs too much shared memory", q));
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, cfg->device) == cudaSuccess) h->num_sms = prop.multiProcessorCount;
        const bool pow2 = is_pow2(M);
        h->finish_on = !env_int("SDRB_NO_FINISH", 0) && pl.rem == 0 && pl.cnt_last == SDRB_TB && q >= pl.edge + 1 &&
                       pow2 && M >= 64 && M <= 1024 && pl.edge + 1 <= 32 && pl.ntiles <= 32 &&
                       (cfg->n_out_sections == 0 || cfg->n_out_sections == 2);
        h->finish_smem = h->finish_on ? finish_smem_bytes(M, pl.edge) : 0;
        if (h->finish_smem > 227 * 1024) h->finish_on = false;
    }
    UP(set_smem_attr(h));
    const size_t dsm = (size_t)M * (2 * sizeof(double2) + sizeof(double));
    pl.demod_in_smem = dsm <= 96 * 1024 ? 1 : 0;
    h->demod_smem = pl.demod_in_smem ? dsm : 0;
    if (h->demod_smem > 48 * 1024)
        if (cudaFuncSetAttribute(is_ssb(cfg->demod) ? k_demod<OUT_SSB> : k_demod<OUT_REAL>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->demod_smem) != cudaSuccess)
            return bail(fail(h, SDRB_ERR_CUDA, "cudaFuncSetAttribute(k_demod) failed"));

    // scratch for max_chunks (seamless: plus the D chunks held back between calls)
    const size_t nch = h->max_chunks + (cfg->seamless ? (size_t)std::max(tab->lookahead, 0) : 0);
    Scratch &sc = h->sc;
    UP(dalloc(h, nch * R * pl.Mf, &sc.ypart));
    UP(dalloc(h, nch * R * nt * 16, &sc.agg));
    UP(dalloc(h, nch * nt, &sc.tile_agg));
    UP(dalloc(h, nch * (nt + 1), &sc.off_tile));
    UP(dalloc(h, nch, &sc.gain));
    UP(dalloc(h, nch, &sc.start));
    UP(dalloc(h, nch * R * (nt + 1) * 16, &sc.carry));
    UP(dalloc(h, nch * R * M, &sc.y));
    UP(dalloc(h, (size_t)1, &sc.iq_state));
    if (cudaMemset(sc.iq_state, 0, sizeof(double2)) != cudaSuccess) return bail(fail(h, SDRB_ERR_CUDA, "memset failed"));
    sc.fftbuf = nullptr; sc.zrow = nullptr; sc.dbg = nullptr; sc.x0 = nullptr;
    if (env_int("SDRB_TC_DEBUG", 0)) {
        UP(dalloc(h, (size_t)64 * 16, &sc.dbg));
        cudaMemset(sc.dbg, 0, 64 * 16 * sizeof(unsigned long long));
    }
    if (!pl.demod_in_smem) {
        UP(dalloc(h, nch * R * 2 * M, &sc.fftbuf));
        UP(dalloc(h, nch * R * M, &sc.zrow));
    }
    UP(setup_tc(h, tab));
    if (cfg->seamless) {
        h->seamless = true;
        SeamDev &sd = h->sd;
        if (pl.rem != 0 || pl.cnt_last != SDRB_TB || tab->lookahead < 1 || !tab->PN || !tab->chunk_step ||
            tab->fs <= 0 || tab->fs >= (1LL << 31) || (cfg->n_out_sections != 0 && cfg->n_out_sections != 2) ||
            (cfg->n_out_sections && (!tab->sos_AM || !tab->sos_CAM || pl.sos_Lseg * 32 != M)))
            return bail(fail(h, SDRB_ERR_ARG, "seamless mode needs the decimation to divide the chunk (q | N), "
                                              "a lookahead >= 1 and its tables"));
        sd.D = tab->lookahead; sd.fs = tab->fs; sd.nedge = pl.edge + 1 + pl.nend;
        UP(upload(h, reinterpret_cast<const long long *>(tab->chunk_step), (size_t)R, &sd.step));
        UP(upload(h, reinterpret_cast<const double2 *>(tab->PN), (size_t)(sd.D + 1) * 8, &sd.PN));
        if (cfg->n_out_sections) {
            for (int i = 0; i < SEAM_NS * SEAM_NS; i++) sd.AM[i] = tab->sos_AM[i];
            UP(upload(h, tab->sos_CAM, (size_t)M * SEAM_NS, &sd.CAM));
        }
        UP(dalloc(h, nch * sd.nedge, &sd.edges));
        UP(dalloc(h, nch * R * 16, &sd.cagg));
        UP(dalloc(h, nch * R * 8, &sd.G));
        UP(dalloc(h, nch * R * 24, &sd.cin));
        UP(dalloc(h, nch * R * (M + 1), &sd.ybuf));
        const size_t sn = (size_t)SEAM_NS * (is_ssb(cfg->demod) ? 2 : 1);   // doubles per SOS state (usb / lsb: complex)
        UP(dalloc(h, nch * R * sn, &sd.echunk));
        UP(dalloc(h, nch * R * sn, &sd.sst));
        UP(dalloc(h, (size_t)R * 8, &sd.fwd));
        UP(dalloc(h, (size_t)R * sn, &sd.sos));
        UP(dalloc(h, (size_t)R * 16, &sd.endv));
        if (cudaMemset(sd.sos, 0, (size_t)R * sn * sizeof(double)) != cudaSuccess)
            return bail(fail(h, SDRB_ERR_CUDA, "memset failed"));
    }
#undef UP
    for (int s = 0; s < 2; s++) {
        if (cudaStreamCreateWithFlags(&h->slot[s].stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->slot[s].done, cudaEventDisableTiming) != cudaSuccess)
            return bail(fail(h, SDRB_ERR_CUDA, "stream/event creation failed"));
    }
    if (cudaEventCreateWithFlags(&h->iq_done, cudaEventDisableTiming) != cudaSuccess)
        return bail(fail(h, SDRB_ERR_CUDA, "event creation failed"));
    *out = h;
    return SDRB_OK;
}

int sdrb_destroy(sdrb_handle *h)
{
    if (!h) return SDRB_OK;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (void *p : h->owned) cudaFree(p);
    for (int s = 0; s < 2; s++) {
        if (h->slot[s].raw) cudaFree(h->slot[s].raw);
        if (h->slot[s].out) cudaFree(h->slot[s].out);
        if (h->slot[s].stream) cudaStreamDestroy(h->slot[s].stream);
        if (h->slot[s].done) cudaEventDestroy(h->slot[s].done);
    }
    if (h->iq_done) cudaEventDestroy(h->iq_done);
    for (int i = 0; i < 5; i++) if (h->pev[i]) cudaEventDestroy(h->pev[i]);
    delete h;
    return SDRB_OK;
}

int sdrb_outputs_per_chunk(const sdrb_handle *h) { return h ? h->pl.M : SDRB_ERR_ARG; }
int sdrb_row_doubles(const sdrb_handle *h) { return h ? h->pl.W : SDRB_ERR_ARG; }
size_t sdrb_chunk_bytes(const sdrb_handle *h) { return h ? (size_t)h->pl.N * 2 * h->pl.itemsize : 0; }
long long sdrb_launch_count(const sdrb_handle *h) { return h ? h->launches : 0; }

int sdrb_process_device(sdrb_handle *h, const void *raw_dev, size_t nchunks, double *out_dev, void *stream)
{
    if (!h || !raw_dev || !out_dev) return fail(h, SDRB_ERR_ARG, "null argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: use sdrb_stream_device / sdrb_stream_end_device");
    if (nchunks == 0) return SDRB_OK;
    if (nchunks > h->max_chunks) return fail(h, SDRB_ERR_ARG, "nchunks %zu > max_chunks %zu", nchunks, h->max_chunks);
    CK(h, cudaSetDevice(h->cfg.device));
    h->last_nchunks = nchunks;
    return launch_chain(h, static_cast<const uint8_t *>(raw_dev), nchunks, out_dev, static_cast<cudaStream_t>(stream));
}

static int ensure_slot(sdrb_handle *h, int s)
{
    Slot &sl = h->slot[s];
    if (!sl.raw) CK(h, cudaMalloc(&sl.raw, h->max_chunks * sdrb_chunk_bytes(h)));
    const size_t och = h->max_chunks + (h->seamless ? (size_t)h->sd.D : 0);
    if (!sl.out) CK(h, cudaMalloc(&sl.out, och * (size_t)h->pl.R * h->pl.W * sizeof(double)));
    return 0;
}

int sdrb_submit(sdrb_handle *h, int s, const void *raw_host, size_t nchunks, double *out_host)
{
    if (!h || !raw_host || !out_host || s < 0 || s > 1) return fail(h, SDRB_ERR_ARG, "bad argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: use sdrb_stream / sdrb_stream_end");
    if (nchunks == 0 || nchunks > h->max_chunks) return fail(h, SDRB_ERR_ARG, "nchunks %zu outside 1..%zu", nchunks, h->max_chunks);
    CK(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_slot(h, s);
    if (rc) return rc;
    Slot &sl = h->slot[s];
    const size_t cb = sdrb_chunk_bytes(h);
    CK(h, cudaMemcpyAsync(sl.raw, raw_host, nchunks * cb, cudaMemcpyHostToDevice, sl.stream));
    // the scratch and the IQ state are shared between slots: kernels of consecutive batches
    // serialise on iq_done, while this batch's H2D overlaps the previous batch's kernels/D2H
    CK(h, cudaStreamWaitEvent(sl.stream, h->iq_done, 0));
    h->last_nchunks = nchunks;
    rc = launch_chain(h, sl.raw, nchunks, sl.out, sl.stream);
    if (rc) return rc;
    CK(h, cudaEventRecord(h->iq_done, sl.stream));
    CK(h, cudaMemcpyAsync(out_host, sl.out, nchunks * (size_t)h->pl.R * h->pl.W * sizeof(double),
                          cudaMemcpyDeviceToHost, sl.stream));
    CK(h, cudaEventRecord(sl.done, sl.stream));
    sl.host_out = out_host; sl.nchunks = nchunks;
    return SDRB_OK;
}

int sdrb_wait(sdrb_handle *h, int s)
{
    if (!h || s < 0 || s > 1) return fail(h, SDRB_ERR_ARG, "bad argument");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->slot[s].stream));
    return SDRB_OK;
}

int sdrb_process(sdrb_handle *h, const void *raw, size_t nchunks, double *out)
{
    if (!h || (!raw && nchunks) || (!out && nchunks)) return fail(h, SDRB_ERR_ARG, "null argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: use sdrb_stream / sdrb_stream_end");
    const size_t cb = sdrb_chunk_bytes(h), W = (size_t)h->pl.W, R = (size_t)h->pl.R;
    if (nchunks <= h->max_chunks) {
        if (nchunks == 0) return SDRB_OK;
        int rc = sdrb_submit(h, 0, raw, nchunks, out);
        if (rc) return rc;
        return sdrb_wait(h, 0);
    }
    // more chunks than one batch holds: rows of `out` are nchunks*W long, so each batch is staged
    // through a per-slot buffer and scattered row by row; the two slots alternate, so the H2D of
    // batch i+1 overlaps the kernels of batch i
    std::vector<double> tmp[2] = {std::vector<double>(h->max_chunks * R * W), std::vector<double>(h->max_chunks * R * W)};
    size_t start[2] = {0, 0}, count[2] = {0, 0};
    auto drain = [&](int s) -> int {
        if (!count[s]) return 0;
        int rc = sdrb_wait(h, s);
        if (rc) return rc;
        for (size_t r = 0; r < R; r++)
            memcpy(out + r * nchunks * W + start[s] * W, tmp[s].data() + r * count[s] * W, count[s] * W * sizeof(double));
        count[s] = 0;
        return 0;
    };
    size_t done = 0;
    int b = 0;
    while (done < nchunks) {
        const int s = b & 1;
        int rc = drain(s);
        if (rc) return rc;
        const size_t n = std::min(h->max_chunks, nchunks - done);
        rc = sdrb_submit(h, s, static_cast<const uint8_t *>(raw) + done * cb, n, tmp[s].data());
        if (rc) return rc;
        start[s] = done; count[s] = n;
        done += n;
        b++;
    }
    int rc = drain(b & 1);
    if (rc) return rc;
    return drain((b + 1) & 1);
}

}  // extern "C"
namespace {
// ------------------------------------------------------------------ seamless streaming
// Copy window slots [from, from + n) to [0, n) of a [slot][per] buffer (from > 0; a slot is never
// read after it has been written when the ranges overlap).
template <typename T>
int seam_shift(sdrb_handle *h, T *buf, size_t per, int from, int n, cudaStream_t st)
{
    if (n <= 0 || from <= 0) return 0;
    if (from >= n) {
        CK(h, cudaMemcpyAsync(buf, buf + (size_t)from * per, (size_t)n * per * sizeof(T), cudaMemcpyDeviceToDevice, st));
    } else {
        for (int j = 0; j < n; j++)
            CK(h, cudaMemcpyAsync(buf + (size_t)j * per, buf + (size_t)(from + j) * per, per * sizeof(T),
                                  cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

// One seamless step: the front end and the IQ kernels over `nch` new chunks (into the window slots
// after the held-back ones), the chunk aggregates and the forward scan; then every chunk that is
// final (all of them when `end`) goes through carry / outputs / demodulation / SOS into `out`.
int seam_step(sdrb_handle *h, const uint8_t *raw, size_t nch, double *out, cudaStream_t st, bool end, size_t *nout)
{
    const DevPlan &pl = h->pl;
    SeamDev &sd = h->sd;
    const int R = pl.R, nt = pl.ntiles, M = pl.M;
    int rc = 0;
    if (nch) {
        const int s0 = h->nwin;
        Scratch base = h->sc, sh = h->sc;
        sh.ypart += (size_t)s0 * R * pl.Mf;
        sh.agg += (size_t)s0 * R * nt * 16;
        sh.tile_agg += (size_t)s0 * nt;
        sh.off_tile += (size_t)s0 * (nt + 1);
        sh.gain += s0;
        sh.start += s0;
        h->sc = sh;
        rc = launch_chain(h, raw, nch, nullptr, st, PH_MAIN | PH_IQSCAN);
        h->sc = base;
        if (rc) return rc;
        rc = with_enc(h, h->enc_code, [&](auto enc) {
            k_seam_edges<decltype(enc)::value><<<(unsigned)nch, 64, 0, st>>>(pl, sd, raw, s0, (int)nch);
            return 0;
        });
        if (rc) return rc;
        const size_t items = nch * (size_t)R;
        k_seam_agg<<<(unsigned)((items + 7) / 8), 256, 0, st>>>(pl, h->sc, sd, s0, (int)nch, h->seen);
        if (h->seen == 0) k_seam_head<<<(unsigned)R, 32, 0, st>>>(pl, h->sc, sd, s0);
        k_seam_fscan<<<(unsigned)R, 256, 0, st>>>(pl, sd, s0, (int)nch);
        h->launches += 3 + (h->seen == 0);
        h->seen += (long long)nch;
        h->nwin += (int)nch;
    }
    long long upto = end ? h->seen : std::max(0LL, h->seen - sd.D);
    const int ne = (int)(upto - h->emitted);
    const long long g0 = h->emitted;
    if (ne > 0) {
        if (end) {
            k_seam_tail<<<(unsigned)R, 32, 0, st>>>(pl, h->sc, sd, h->nwin - 1, h->seen - 1);
            h->launches++;
        }
        const size_t items = (size_t)ne * R;
        const unsigned wg = (unsigned)((items + 7) / 8);
        k_seam_carry<<<wg, 256, 0, st>>>(pl, h->sc, sd, ne, h->nwin, g0, end ? 1 : 0);
        k_seam_y<<<wg, 256, 0, st>>>(pl, h->sc, sd, ne, h->nwin, g0, end ? 1 : 0);
        const bool ssb = is_ssb(pl.demod);
        if (ssb) k_seam_demod<true><<<wg, 256, 0, st>>>(pl, sd, out, ne, h->nwin, end ? 1 : 0);
        else k_seam_demod<false><<<wg, 256, 0, st>>>(pl, sd, out, ne, h->nwin, end ? 1 : 0);
        h->launches += 3;
        if (pl.nsec_out) {
            const size_t total = items * M;
            const unsigned fg = (unsigned)std::min<size_t>((total + 255) / 256, (size_t)h->num_sms * 16);
            if (ssb) {
                k_seam_sscan<double2><<<(unsigned)R, 32, 0, st>>>(pl, sd, ne);
                k_seam_frame<true><<<fg, 256, 0, st>>>(pl, sd, out, ne);
            } else {
                k_seam_sscan<double><<<(unsigned)R, 32, 0, st>>>(pl, sd, ne);
                k_seam_frame<false><<<fg, 256, 0, st>>>(pl, sd, out, ne);
            }
            h->launches += 2;
        }
        CK(h, cudaGetLastError());
        // the chunks still held back move to the front of the window
        const int keep = h->nwin - ne;
        if ((rc = seam_shift(h, h->sc.ypart, (size_t)R * pl.Mf, ne, keep, st)) ||
            (rc = seam_shift(h, h->sc.agg, (size_t)R * nt * 16, ne, keep, st)) ||
            (rc = seam_shift(h, h->sc.off_tile, (size_t)(nt + 1), ne, keep, st)) ||
            (rc = seam_shift(h, sd.edges, (size_t)sd.nedge, ne, keep, st)) ||
            (rc = seam_shift(h, sd.cagg, (size_t)R * 16, ne, keep, st)) ||
            (rc = seam_shift(h, sd.G, (size_t)R * 8, ne, keep, st)))
            return rc;
        h->nwin = keep;
        h->emitted = upto;
    }
    CK(h, cudaGetLastError());
    if (nout) *nout = (size_t)std::max(ne, 0);
    if (end) {   // a new stream starts from scratch: counters, output filter and IQ corrector
        h->seen = h->emitted = 0;
        h->nwin = 0;
        CK(h, cudaMemsetAsync(sd.sos, 0, (size_t)R * SEAM_NS * (is_ssb(pl.demod) ? 2 : 1) * sizeof(double), st));
        CK(h, cudaMemsetAsync(h->sc.iq_state, 0, sizeof(double2), st));
    }
    return 0;
}
}  // namespace
extern "C" {

int sdrb_stream_device(sdrb_handle *h, const void *raw_dev, size_t nchunks, double *out_dev, void *stream,
                       size_t *nchunks_out)
{
    if (nchunks_out) *nchunks_out = 0;
    if (!h || (!raw_dev && nchunks) || !out_dev) return fail(h, SDRB_ERR_ARG, "null argument");
    if (!h->seamless) return fail(h, SDRB_ERR_STATE, "sdrb_stream needs a handle created with cfg.seamless");
    if (nchunks > h->max_chunks) return fail(h, SDRB_ERR_ARG, "nchunks %zu > max_chunks %zu", nchunks, h->max_chunks);
    if (h->pl.demod == SDRB_IQ && ((uintptr_t)out_dev & 15))
        return fail(h, SDRB_ERR_ARG, "iq output is stored as 16-byte (Re, Im) pairs: `out` must be 16-byte aligned");
    CK(h, cudaSetDevice(h->cfg.device));
    return seam_step(h, static_cast<const uint8_t *>(raw_dev), nchunks, out_dev, static_cast<cudaStream_t>(stream), false,
                     nchunks_out);
}

int sdrb_stream_end_device(sdrb_handle *h, double *out_dev, void *stream, size_t *nchunks_out)
{
    if (nchunks_out) *nchunks_out = 0;
    if (!h || !out_dev) return fail(h, SDRB_ERR_ARG, "null argument");
    if (!h->seamless) return fail(h, SDRB_ERR_STATE, "sdrb_stream_end needs a handle created with cfg.seamless");
    if (h->pl.demod == SDRB_IQ && ((uintptr_t)out_dev & 15))
        return fail(h, SDRB_ERR_ARG, "iq output is stored as 16-byte (Re, Im) pairs: `out` must be 16-byte aligned");
    CK(h, cudaSetDevice(h->cfg.device));
    return seam_step(h, nullptr, 0, out_dev, static_cast<cudaStream_t>(stream), true, nchunks_out);
}

static int seam_host(sdrb_handle *h, const void *raw_host, size_t nchunks, double *out_host, size_t *nchunks_out, bool end)
{
    if (nchunks_out) *nchunks_out = 0;
    if (!h || (!raw_host && nchunks) || !out_host) return fail(h, SDRB_ERR_ARG, "null argument");
    if (!h->seamless) return fail(h, SDRB_ERR_STATE, "sdrb_stream needs a handle created with cfg.seamless");
    if (nchunks > h->max_chunks) return fail(h, SDRB_ERR_ARG, "nchunks %zu > max_chunks %zu", nchunks, h->max_chunks);
    CK(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_slot(h, 0);
    if (rc) return rc;
    Slot &sl = h->slot[0];
    if (nchunks)
        CK(h, cudaMemcpyAsync(sl.raw, raw_host, nchunks * sdrb_chunk_bytes(h), cudaMemcpyHostToDevice, sl.stream));
    size_t ne = 0;
    rc = seam_step(h, sl.raw, nchunks, sl.out, sl.stream, end, &ne);
    if (rc) return rc;
    if (ne)
        CK(h, cudaMemcpyAsync(out_host, sl.out, ne * (size_t)h->pl.R * h->pl.W * sizeof(double), cudaMemcpyDeviceToHost,
                              sl.stream));
    CK(h, cudaStreamSynchronize(sl.stream));
    if (nchunks_out) *nchunks_out = ne;
    return SDRB_OK;
}

int sdrb_stream(sdrb_handle *h, const void *raw_host, size_t nchunks, double *out_host, size_t *nchunks_out)
{
    return seam_host(h, raw_host, nchunks, out_host, nchunks_out, false);
}

int sdrb_stream_end(sdrb_handle *h, double *out_host, size_t *nchunks_out)
{
    return seam_host(h, nullptr, 0, out_host, nchunks_out, true);
}

int sdrb_stream_lookahead(const sdrb_handle *h)
{
    if (!h) return SDRB_ERR_ARG;
    return h->seamless ? h->sd.D : 0;
}

int sdrb_set_smooth(sdrb_handle *h, int window, int nhead, int ntail, int lo, const double *tab)
{
    if (!h || window < 0 || (window > 0 && (!tab || nhead < 0 || ntail < 0 || nhead + ntail > h->pl.M)))
        return fail(h, SDRB_ERR_ARG, "bad argument");
    if (h->seamless && window > 0)
        return fail(h, SDRB_ERR_ARG, "--smooth-output is per-chunk Savitzky-Golay by definition: not available in seamless mode");
    if (h->pl.demod == SDRB_IQ && window > 0)
        return fail(h, SDRB_ERR_ARG, "--smooth-output is not available with iq output (complex baseband is not smoothed)");
    if (window > h->pl.M) return fail(h, SDRB_ERR_ARG, "smoothing window %d longer than a chunk's %d outputs", window, h->pl.M);
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaDeviceSynchronize());
    h->smooth_w = 0;
    if (window == 0) return SDRB_OK;
    const size_t n = (size_t)(nhead + 1 + ntail) * window;
    double *dS = nullptr;
    int rc = dalloc(h, n, &dS);
    if (rc) return rc;
    CK(h, cudaMemcpy(dS, tab, n * sizeof(double), cudaMemcpyHostToDevice));
    if (!h->smooth_tmp) {
        rc = dalloc(h, h->max_chunks * (size_t)h->pl.R * h->pl.M, &h->smooth_tmp);
        if (rc) return rc;
    }
    h->smooth_S = dS;
    h->smooth_nhead = nhead; h->smooth_ntail = ntail; h->smooth_lo = lo;
    h->smooth_w = window;
    return SDRB_OK;
}

int sdrb_iq_gain(sdrb_handle *h, const void *raw_host, size_t nchunks)
{
    if (!h || !raw_host) return fail(h, SDRB_ERR_ARG, "null argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: the IQ state advances with sdrb_stream");
    if (nchunks == 0 || !h->pl.correct_iq) return SDRB_OK;
    if (nchunks > h->max_chunks) return fail(h, SDRB_ERR_ARG, "nchunks %zu > max_chunks %zu", nchunks, h->max_chunks);
    CK(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_slot(h, 0);
    if (rc) return rc;
    Slot &sl = h->slot[0];
    CK(h, cudaMemcpyAsync(sl.raw, raw_host, nchunks * sdrb_chunk_bytes(h), cudaMemcpyHostToDevice, sl.stream));
    CK(h, cudaStreamWaitEvent(sl.stream, h->iq_done, 0));
    rc = with_enc(h, h->enc_code, [&](auto enc) {
        k_iqchunk<decltype(enc)::value><<<(unsigned)((nchunks + 7) / 8), 256, 0, sl.stream>>>(h->pl, h->sc, sl.raw, (int)nchunks);
        return 0;
    });
    if (rc) return rc;
    k_iqscan_c<<<1, 1024, 0, sl.stream>>>(h->pl, h->sc, (int)nchunks);
    h->launches += 2;
    CK(h, cudaGetLastError());
    CK(h, cudaEventRecord(h->iq_done, sl.stream));
    CK(h, cudaStreamSynchronize(sl.stream));
    return SDRB_OK;
}

int sdrb_process_device_phases(sdrb_handle *h, const void *raw_dev, size_t nchunks, double *out_dev, void *stream, int phases)
{
    if (!h || !raw_dev || (!out_dev && (phases & PH_FINISH))) return fail(h, SDRB_ERR_ARG, "null argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: time-segment phases are not available");
    if (nchunks == 0) return SDRB_OK;
    if (nchunks > h->max_chunks) return fail(h, SDRB_ERR_ARG, "nchunks %zu > max_chunks %zu", nchunks, h->max_chunks);
    CK(h, cudaSetDevice(h->cfg.device));
    h->last_nchunks = nchunks;
    if (phases & SDRB_PHASE_ZERO_IQ)
        CK(h, cudaMemsetAsync(h->sc.iq_state, 0, sizeof(double2), static_cast<cudaStream_t>(stream)));
    return launch_chain(h, static_cast<const uint8_t *>(raw_dev), nchunks, out_dev, static_cast<cudaStream_t>(stream), phases & 7);
}

int sdrb_iq_export_device(sdrb_handle *h, double *dst3_dev, double nsamples, void *stream)
{
    if (!h || !dst3_dev) return fail(h, SDRB_ERR_ARG, "null argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: time-segment phases are not available");
    CK(h, cudaSetDevice(h->cfg.device));
    k_iq_export<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(h->sc, dst3_dev, nsamples);
    h->launches++;
    CK(h, cudaGetLastError());
    return SDRB_OK;
}

int sdrb_iq_prefix_device(sdrb_handle *h, const double *gains3_dev, int rank, void *stream)
{
    if (!h || !gains3_dev || rank < 0) return fail(h, SDRB_ERR_ARG, "bad argument");
    if (h->seamless) return fail(h, SDRB_ERR_STATE, "seamless handle: time-segment phases are not available");
    CK(h, cudaSetDevice(h->cfg.device));
    k_iq_prefix<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(h->sc, gains3_dev, rank, h->pl.lam);
    h->launches++;
    CK(h, cudaGetLastError());
    return SDRB_OK;
}

int sdrb_set_profiling(sdrb_handle *h, int on)
{
    if (!h) return fail(h, SDRB_ERR_ARG, "null argument");
    CK(h, cudaSetDevice(h->cfg.device));
    if (on) for (int i = 0; i < 5; i++) if (!h->pev[i]) CK(h, cudaEventCreate(&h->pev[i]));
    h->profiling = on != 0;
    return SDRB_OK;
}

int sdrb_kernel_times(sdrb_handle *h, float ms[4])
{
    if (!h || !ms) return fail(h, SDRB_ERR_ARG, "null argument");
    for (int i = 0; i < 5; i++) if (!h->pev_valid[i]) return fail(h, SDRB_ERR_STATE, "no profiled batch");
    CK(h, cudaEventSynchronize(h->pev[4]));
    for (int i = 0; i < 4; i++) CK(h, cudaEventElapsedTime(&ms[i], h->pev[i], h->pev[i + 1]));
    return SDRB_OK;
}

int sdrb_get_iq_state(sdrb_handle *h, double off[2])
{
    if (!h || !off) return fail(h, SDRB_ERR_ARG, "null argument");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(off, h->sc.iq_state, sizeof(double2), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_set_iq_state(sdrb_handle *h, const double off[2])
{
    if (!h || !off) return fail(h, SDRB_ERR_ARG, "null argument");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(h->sc.iq_state, off, sizeof(double2), cudaMemcpyHostToDevice));
    return SDRB_OK;
}

/* diagnostic: k_tc pipeline timeline of CTA 0 (clock64 per event), needs SDRB_TC_DEBUG=1 at create */
int sdrb_read_debug(sdrb_handle *h, unsigned long long *out1024)
{
    if (!h || !out1024 || !h->sc.dbg) return fail(h, SDRB_ERR_STATE, "no debug buffer");
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(out1024, h->sc.dbg, 64 * 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_reserve_sms(sdrb_handle *h, int nsm)
{
    if (!h || nsm < 0 || nsm >= h->num_sms) return fail(h, SDRB_ERR_ARG, "bad argument");
    h->reserved_sms = nsm;
    return SDRB_OK;
}

int sdrb_keep_decimated(sdrb_handle *h, int on)
{
    if (!h) return fail(h, SDRB_ERR_ARG, "null argument");
    h->keep_y = on != 0;
    return SDRB_OK;
}

int sdrb_read_decimated(sdrb_handle *h, size_t nchunks, double *y_host)
{
    if (!h || !y_host) return fail(h, SDRB_ERR_ARG, "null argument");
    if (h->finish_on && !h->keep_y) return fail(h, SDRB_ERR_STATE, "decimator output not kept: call sdrb_keep_decimated(h, 1) first");
    if (nchunks > h->last_nchunks) return fail(h, SDRB_ERR_STATE, "only %zu chunks in the last batch", h->last_nchunks);
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(y_host, h->sc.y, nchunks * (size_t)h->pl.R * h->pl.M * sizeof(double2), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- module-level operators
namespace {
// device allocation freed on every exit path
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <typename T> T *as() const { return static_cast<T *>(p); }
};

// The plot feeds are called once per displayed frame on a few hundred kilobytes: their device and
// page-locked staging buffers are kept between calls (cudaMalloc / cudaFree cost more than the
// transform).  One set per device and slot, grown on demand, never shrunk; calls are serialised.
struct FeedWorkspace {
    static constexpr int kSlots = 6, kMaxDev = 16;
    void *dev[kMaxDev][kSlots] = {};
    size_t dev_cap[kMaxDev][kSlots] = {};
    void *host[kMaxDev][2] = {};
    size_t host_cap[kMaxDev][2] = {};
    std::mutex mu;
    cudaError_t get(int device, int slot, size_t bytes, void **out)
    {
        if (dev_cap[device][slot] < bytes) {
            if (dev[device][slot]) cudaFree(dev[device][slot]);
            dev[device][slot] = nullptr; dev_cap[device][slot] = 0;
            cudaError_t e = cudaMalloc(&dev[device][slot], bytes);
            if (e != cudaSuccess) return e;
            dev_cap[device][slot] = bytes;
        }
        *out = dev[device][slot];
        return cudaSuccess;
    }
    cudaError_t get_host(int device, int slot, size_t bytes, void **out)
    {
        if (host_cap[device][slot] < bytes) {
            if (host[device][slot]) cudaFreeHost(host[device][slot]);
            host[device][slot] = nullptr; host_cap[device][slot] = 0;
            cudaError_t e = cudaHostAlloc(&host[device][slot], bytes, cudaHostAllocDefault);
            if (e != cudaSuccess) return e;
            host_cap[device][slot] = bytes;
        }
        *out = host[device][slot];
        return cudaSuccess;
    }
};
FeedWorkspace g_feed;

int need_device(int device)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, SDRB_ERR_CUDA, "no CUDA device: libsdrterm_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, SDRB_ERR_ARG, "bad device ordinal");
    CK(nullptr, cudaSetDevice(device));
    return 0;
}

// scipy.signal.resample(r, M) of a real row of h samples as a dense [M][h] matrix (any h, any
// M >= h): y[k] = sum_m W[k][m] r[m], W[k][m] = (1/h) (1 + 2 sum_{b=1}^{B} c_b cos(b theta)),
// theta = 2 pi (k/M - m/h), B = floor(h/2), c_B = 1/2 when h is even and M > h (the unpaired
// bin is split), closed form of the cosine sum in long double.
std::vector<double> resample_matrix(int h, int M)
{
    std::vector<double> W((size_t)M * h);
    const long double two_pi = 6.283185307179586476925286766559005768L;
    const int B = h / 2;
    const bool split = (h % 2 == 0) && M > h;
    const int nfull = split ? B - 1 : B;                 // bins with weight 1
    for (int k = 0; k < M; k++)
        for (int m = 0; m < h; m++) {
            // reduce the angle exactly in integers first: theta = 2 pi (k h - m M) / (M h)
            const long long num = ((long long)k * h - (long long)m * M) % ((long long)M * h);
            const long double th = two_pi * (long double)num / ((long double)M * (long double)h);
            long double s;
            const long double sh = sinl(th / 2);
            if (fabsl(sh) < 1e-18L) s = (long double)nfull;
            else s = sinl(nfull * th / 2) * cosl((nfull + 1) * th / 2) / sh;   // sum_{b=1}^{nfull} cos(b th)
            long double v = 1.0L + 2.0L * s;
            if (split) v += cosl(B * th);                // 2 * (1/2) * cos(B th)
            W[(size_t)k * h + m] = (double)(v / h);
        }
    return W;
}
}  // namespace

extern "C" {

static int demod_op(int device, const double *y, int R, int M, double *out, int demod)
{
    if (!y || !out || R < 1 || M < 1) return fail(nullptr, SDRB_ERR_ARG, "bad argument");
    int rc = need_device(device);
    if (rc) return rc;
    DevPlan pl{};
    pl.M = M; pl.R = R; pl.nsec_out = 0;
    pl.W = demod == SDRB_IQ ? 2 * M : M;
    const int h2 = M >> 1;
    pl.fft_ok = (M == 2 * h2) && is_pow2(h2);
    pl.fft_n = pl.fft_ok ? M : 0;
    if (demod == SDRB_FM && (M & 1))
        return fail(nullptr, SDRB_ERR_ARG, "fmDemod pairs samples: the row length must be even (got %d)", M);
    std::vector<double2> tw = make_twiddles(pl.fft_n);
    DevBuf d_tw, d_y, d_out, d_fft, d_z, d_w;
    const size_t dsm = (size_t)M * (2 * sizeof(double2) + sizeof(double));
    pl.demod_in_smem = dsm <= 48 * 1024;
    CK(nullptr, d_tw.alloc(tw.size() * sizeof(double2)));
    CK(nullptr, d_y.alloc((size_t)R * M * sizeof(double2)));
    CK(nullptr, d_out.alloc((size_t)R * pl.W * sizeof(double)));
    if (!pl.demod_in_smem) {
        CK(nullptr, d_fft.alloc((size_t)R * 2 * M * sizeof(double2)));
        CK(nullptr, d_z.alloc((size_t)R * M * sizeof(double)));
    }
    if (demod == SDRB_FM && !pl.fft_ok) {
        // any even length: the same dense interpolation the engine uses for non-FFT sizes
        const std::vector<double> W = resample_matrix(h2, M);
        CK(nullptr, d_w.alloc(W.size() * sizeof(double)));
        CK(nullptr, cudaMemcpy(d_w.p, W.data(), W.size() * sizeof(double), cudaMemcpyHostToDevice));
        pl.fm_interp = d_w.as<double>();
    }
    CK(nullptr, cudaMemcpy(d_tw.p, tw.data(), tw.size() * sizeof(double2), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(d_y.p, y, (size_t)R * M * sizeof(double2), cudaMemcpyHostToDevice));
    pl.tw = d_tw.as<double2>();
    // rows are laid out [R][M]: run as R "rows" of a single chunk
    if (demod == SDRB_IQ)
        k_demod<OUT_IQ><<<R, 128, 0>>>(pl, d_y.as<double2>(), d_out.as<double>(), nullptr, nullptr, 1, demod, 0, 0);
    else
        k_demod<OUT_REAL><<<R, 128, pl.demod_in_smem ? dsm : 0>>>(pl, d_y.as<double2>(), d_out.as<double>(), d_fft.as<double2>(),
                                                                  d_z.as<double>(), 1, demod, 0, 0);
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaDeviceSynchronize());
    CK(nullptr, cudaMemcpy(out, d_out.p, (size_t)R * pl.W * sizeof(double), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_fm_demod(int device, const double *y, int R, int M, double *out) { return demod_op(device, y, R, M, out, SDRB_FM); }
int sdrb_am_demod(int device, const double *y, int R, int M, double *out) { return demod_op(device, y, R, M, out, SDRB_AM); }
int sdrb_real_output(int device, const double *y, int R, int M, double *out) { return demod_op(device, y, R, M, out, SDRB_RE); }
int sdrb_imag_output(int device, const double *y, int R, int M, double *out) { return demod_op(device, y, R, M, out, SDRB_IM); }
int sdrb_iq_output(int device, const double *y, int R, int M, double *out) { return demod_op(device, y, R, M, out, SDRB_IQ); }

int sdrb_ssb_demod(int device, const double *y, int R, int M, const double *sos, int nsec, double omega, double *out)
{
    if (!y || !out || !sos || R < 1 || M < 1 || nsec < 1 || nsec > 4) return fail(nullptr, SDRB_ERR_ARG, "bad argument");
    if (!(std::fabs(omega) > 0.0) || !(std::fabs(omega) < M_PI / 2))
        return fail(nullptr, SDRB_ERR_ARG, "ssb rotation %g outside 0 < |omega| < pi/2", omega);
    for (int s = 0; s < nsec; s++)
        if (sos[6 * s + 3] != 1.0) return fail(nullptr, SDRB_ERR_ARG, "sos section %d is not normalised (a0 != 1)", s);
    int rc = need_device(device);
    if (rc) return rc;
    DevPlan pl{};
    pl.M = pl.W = M; pl.R = R; pl.nsec_out = nsec; pl.sos_ns = 2 * nsec; pl.sos_Lseg = (M + 31) / 32;
    pl.ssb_omega = omega;
    for (int i = 0; i < 6 * nsec; i++) pl.out_sos[i] = sos[i];
    // the prototype's state space (A, c) in extended precision -- the same DF2T state variables as
    // plan.py's _cascade_state_space -- then A^Lseg and its squarings, c A^i (i < Lseg) and
    // e^{j omega k} (k <= M)
    const int ns = pl.sos_ns, Ls = pl.sos_Lseg;
    std::vector<long double> A((size_t)ns * ns, 0.0L), cvec(ns, 0.0L);
    {
        std::vector<long double> u(ns + 1, 0.0L);
        u[ns] = 1.0L;
        for (int k = 0; k < nsec; k++) {
            const long double b0 = sos[6 * k], b1 = sos[6 * k + 1], b2 = sos[6 * k + 2], a1 = sos[6 * k + 4], a2 = sos[6 * k + 5];
            std::vector<long double> yv(ns + 1), z0(ns + 1), z1(ns + 1);
            for (int j = 0; j <= ns; j++) yv[j] = b0 * u[j];
            yv[2 * k] += 1.0L;
            for (int j = 0; j <= ns; j++) { z0[j] = b1 * u[j] - a1 * yv[j]; z1[j] = b2 * u[j] - a2 * yv[j]; }
            z0[2 * k + 1] += 1.0L;
            for (int j = 0; j < ns; j++) { A[(size_t)(2 * k) * ns + j] = z0[j]; A[(size_t)(2 * k + 1) * ns + j] = z1[j]; }
            u = yv;
        }
        for (int j = 0; j < ns; j++) cvec[j] = u[j];
    }
    std::vector<double> ca((size_t)Ls * ns);
    std::vector<long double> P((size_t)ns * ns, 0.0L), cur = cvec;
    for (int i = 0; i < ns; i++) P[(size_t)i * ns + i] = 1.0L;
    for (int i = 0; i < Ls; i++) {
        for (int j = 0; j < ns; j++) ca[(size_t)i * ns + j] = (double)cur[j];
        std::vector<long double> nx(ns, 0.0L), NP((size_t)ns * ns, 0.0L);
        for (int j = 0; j < ns; j++)
            for (int b = 0; b < ns; b++) nx[j] += cur[b] * A[(size_t)b * ns + j];
        for (int a = 0; a < ns; a++)
            for (int b = 0; b < ns; b++)
                for (int k = 0; k < ns; k++) NP[(size_t)a * ns + b] += A[(size_t)a * ns + k] * P[(size_t)k * ns + b];
        cur = nx;
        P = NP;
    }
    for (int lv = 0; lv < 5; lv++) {                                      // (A^Lseg)^(2^lv)
        for (int i = 0; i < ns * ns; i++) pl.sos_AP[lv * ns * ns + i] = (double)P[i];
        std::vector<long double> PP((size_t)ns * ns, 0.0L);
        for (int a = 0; a < ns; a++)
            for (int b = 0; b < ns; b++)
                for (int k = 0; k < ns; k++) PP[(size_t)a * ns + b] += P[(size_t)a * ns + k] * P[(size_t)k * ns + b];
        P = PP;
    }
    std::vector<double2> rot((size_t)M + 1);
    for (int k = 0; k <= M; k++) {
        const long double a = (long double)omega * (long double)k;
        rot[k] = make_double2((double)cosl(a), (double)sinl(a));
    }
    DevBuf d_y, d_out, d_fft, d_z, d_ca, d_rot;
    const size_t dsm = (size_t)M * (2 * sizeof(double2) + sizeof(double));
    pl.demod_in_smem = dsm <= 48 * 1024;
    CK(nullptr, d_y.alloc((size_t)R * M * sizeof(double2)));
    CK(nullptr, d_out.alloc((size_t)R * M * sizeof(double)));
    CK(nullptr, d_ca.alloc(ca.size() * sizeof(double)));
    CK(nullptr, d_rot.alloc(rot.size() * sizeof(double2)));
    if (!pl.demod_in_smem) {
        CK(nullptr, d_fft.alloc((size_t)R * 2 * M * sizeof(double2)));
        CK(nullptr, d_z.alloc((size_t)R * M * sizeof(double)));
    }
    CK(nullptr, cudaMemcpy(d_y.p, y, (size_t)R * M * sizeof(double2), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(d_ca.p, ca.data(), ca.size() * sizeof(double), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(d_rot.p, rot.data(), rot.size() * sizeof(double2), cudaMemcpyHostToDevice));
    pl.sos_CA = d_ca.as<double>();
    pl.ssb_rot = d_rot.as<double2>();
    // rows are laid out [R][M]: run as R "rows" of a single chunk
    k_demod<OUT_SSB><<<R, 128, pl.demod_in_smem ? dsm : 0>>>(pl, d_y.as<double2>(), d_out.as<double>(), d_fft.as<double2>(),
                                                             d_z.as<double>(), 1, SDRB_USB, 1, 0);
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaDeviceSynchronize());
    CK(nullptr, cudaMemcpy(out, d_out.p, (size_t)R * M * sizeof(double), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_shift_freq(int device, const double *y, const double *shift, int R, int N, double *res)
{
    if (!y || !shift || !res || R < 1 || N < 1) return fail(nullptr, SDRB_ERR_ARG, "bad argument");
    int rc = need_device(device);
    if (rc) return rc;
    DevBuf d_y, d_s, d_r;
    CK(nullptr, d_y.alloc((size_t)N * sizeof(double2)));
    CK(nullptr, d_s.alloc((size_t)R * N * sizeof(double2)));
    CK(nullptr, d_r.alloc((size_t)R * N * sizeof(double2)));
    CK(nullptr, cudaMemcpy(d_y.p, y, (size_t)N * sizeof(double2), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(d_s.p, shift, (size_t)R * N * sizeof(double2), cudaMemcpyHostToDevice));
    k_shift<<<148 * 4, 256>>>(d_y.as<double2>(), d_s.as<double2>(), d_r.as<double2>(), R, N);
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaDeviceSynchronize());
    CK(nullptr, cudaMemcpy(res, d_r.p, (size_t)R * N * sizeof(double2), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_power_spectrum(int device, const double *y, const double *shift, int N, int batch, double *out)
{
    if (!y || !out || batch < 1 || N < 4 || (N & (N - 1))) return fail(nullptr, SDRB_ERR_ARG, "power spectrum: N must be a power of two >= 4");
    int rc = need_device(device);
    if (rc) return rc;
    if (device >= FeedWorkspace::kMaxDev) return fail(nullptr, SDRB_ERR_ARG, "bad device ordinal");
    std::lock_guard<std::mutex> lock(g_feed.mu);
    const size_t nb = (size_t)batch * N * sizeof(double2), nout = (size_t)batch * N * sizeof(double);
    void *pa, *pb, *ps = nullptr, *po, *hin, *hout;
    CK(nullptr, g_feed.get(device, 0, nb, &pa));
    CK(nullptr, g_feed.get(device, 1, nb, &pb));
    CK(nullptr, g_feed.get(device, 2, nout, &po));
    CK(nullptr, g_feed.get_host(device, 0, nb + (size_t)N * sizeof(double2), &hin));
    CK(nullptr, g_feed.get_host(device, 1, nout, &hout));
    // pageable -> page-locked on the host, then asynchronous copies and kernels on one stream
    std::memcpy(hin, y, nb);
    CK(nullptr, cudaMemcpyAsync(pa, hin, nb, cudaMemcpyHostToDevice, 0));
    const double2 *sh = nullptr;
    if (shift) {
        CK(nullptr, g_feed.get(device, 3, (size_t)N * sizeof(double2), &ps));
        std::memcpy(static_cast<char *>(hin) + nb, shift, (size_t)N * sizeof(double2));
        CK(nullptr, cudaMemcpyAsync(ps, static_cast<char *>(hin) + nb, (size_t)N * sizeof(double2), cudaMemcpyHostToDevice, 0));
        sh = static_cast<const double2 *>(ps);
    }
    double2 *src = static_cast<double2 *>(pa), *dst = static_cast<double2 *>(pb);
    const dim3 grid4((unsigned)std::min(148 * 8, (N / 4 + 255) / 256), (unsigned)batch);
    int Ns = 1;
    for (; Ns * 4 <= N; Ns <<= 2) {
        k_gfft4<<<grid4, 256>>>(src, dst, sh, N, Ns);
        sh = nullptr;
        std::swap(src, dst);
    }
    if (Ns < N) {
        k_gfft2<<<grid4, 256>>>(src, dst, sh, N, Ns);
        std::swap(src, dst);
    }
    k_spectrum_db<<<dim3((unsigned)std::min(148 * 8, (N + 255) / 256), (unsigned)batch), 256>>>(src, static_cast<double *>(po), N);
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaMemcpyAsync(hout, po, nout, cudaMemcpyDeviceToHost, 0));
    CK(nullptr, cudaStreamSynchronize(0));
    std::memcpy(out, hout, nout);
    return SDRB_OK;
}

int sdrb_stft_db(int device, const double *y, const double *shift, int n, const double *win, int nperseg, int hop,
                 int mfft, int p_num, double *out)
{
    if (!y || !win || !out || n < 1 || nperseg < 1 || hop < 1 || p_num < 1 || mfft < nperseg || mfft < 4 || mfft > 4096 ||
        (mfft & (mfft - 1)))
        return fail(nullptr, SDRB_ERR_ARG, "stft: mfft must be a power of two in 4..4096 and >= nperseg");
    int rc = need_device(device);
    if (rc) return rc;
    if (device >= FeedWorkspace::kMaxDev) return fail(nullptr, SDRB_ERR_ARG, "bad device ordinal");
    std::lock_guard<std::mutex> lock(g_feed.mu);
    const size_t ny = (size_t)n * sizeof(double2), nw = (size_t)nperseg * sizeof(double), nout = (size_t)mfft * p_num * sizeof(double);
    void *py, *ps = nullptr, *pw, *po, *hin, *hout;
    CK(nullptr, g_feed.get(device, 0, ny, &py));
    CK(nullptr, g_feed.get(device, 4, nw, &pw));
    CK(nullptr, g_feed.get(device, 5, nout, &po));
    CK(nullptr, g_feed.get_host(device, 0, 2 * ny + nw, &hin));
    CK(nullptr, g_feed.get_host(device, 1, nout, &hout));
    char *h8 = static_cast<char *>(hin);
    std::memcpy(h8, y, ny);
    std::memcpy(h8 + 2 * ny, win, nw);
    CK(nullptr, cudaMemcpyAsync(py, h8, ny, cudaMemcpyHostToDevice, 0));
    CK(nullptr, cudaMemcpyAsync(pw, h8 + 2 * ny, nw, cudaMemcpyHostToDevice, 0));
    const double2 *sh = nullptr;
    if (shift) {
        CK(nullptr, g_feed.get(device, 3, ny, &ps));
        std::memcpy(h8 + ny, shift, ny);
        CK(nullptr, cudaMemcpyAsync(ps, h8 + ny, ny, cudaMemcpyHostToDevice, 0));
        sh = static_cast<const double2 *>(ps);
    }
    const int W = 4;
    const size_t smem = ((size_t)(mfft >> 1) + (size_t)W * 2 * mfft) * sizeof(double2);
    static size_t smem_set = 0;
    if (smem > smem_set) {
        CK(nullptr, cudaFuncSetAttribute(k_stft_db, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
    }
    const unsigned grid = (unsigned)std::min(148 * 2, (p_num + W - 1) / W);
    k_stft_db<<<grid, 32 * W, smem>>>(static_cast<const double2 *>(py), sh, static_cast<const double *>(pw), static_cast<double *>(po),
                                      n, nperseg, hop, nperseg / 2, mfft, p_num);
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaMemcpyAsync(hout, po, nout, cudaMemcpyDeviceToHost, 0));
    CK(nullptr, cudaStreamSynchronize(0));
    std::memcpy(out, hout, nout);
    return SDRB_OK;
}

int sdrb_decode_iq(int device, const void *raw, size_t nsamples, char enc, int swap, double *z_out)
{
    const int code = enc_code_of(enc);
    if (!raw || !z_out || code < 0 || code == ENC_Z) return fail(nullptr, SDRB_ERR_ARG, "bad argument");
    if (nsamples == 0) return SDRB_OK;
    int rc = need_device(device);
    if (rc) return rc;
    const size_t nbytes = nsamples * 2 * (size_t)itemsize_of(code);
    DevBuf d_raw, d_z;
    CK(nullptr, d_raw.alloc(nbytes));
    CK(nullptr, d_z.alloc(nsamples * sizeof(double2)));
    CK(nullptr, cudaMemcpy(d_raw.p, raw, nbytes, cudaMemcpyHostToDevice));
    const unsigned grid = (unsigned)std::min<size_t>((nsamples + 255) / 256, 148 * 8);
    const uint8_t *r8 = d_raw.as<uint8_t>();
    double2 *z = d_z.as<double2>();
    rc = with_enc(nullptr, code, [&](auto enc) {
        constexpr int E = decltype(enc)::value;
        if constexpr (E != ENC_Z) k_decode<E><<<grid, 256>>>(r8, z, nsamples, swap);   // ENC_Z is refused above
        return 0;
    });
    if (rc) return rc;
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaDeviceSynchronize());
    CK(nullptr, cudaMemcpy(z_out, d_z.p, nsamples * sizeof(double2), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_correct_iq(int device, double *z_inout, size_t nsamples, double off_inout[2], double L)
{
    if (!z_inout || !off_inout) return fail(nullptr, SDRB_ERR_ARG, "null argument");
    if (nsamples == 0) return SDRB_OK;
    int rc = need_device(device);
    if (rc) return rc;
    DevBuf d_z, d_off;
    CK(nullptr, d_z.alloc(nsamples * sizeof(double2)));
    CK(nullptr, d_off.alloc(sizeof(double2)));
    CK(nullptr, cudaMemcpy(d_z.p, z_inout, nsamples * sizeof(double2), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(d_off.p, off_inout, sizeof(double2), cudaMemcpyHostToDevice));
    k_correct_iq<<<1, 1024>>>(d_z.as<double2>(), nsamples, d_off.as<double2>(), L);
    CK(nullptr, cudaGetLastError());
    CK(nullptr, cudaDeviceSynchronize());
    CK(nullptr, cudaMemcpy(z_inout, d_z.p, nsamples * sizeof(double2), cudaMemcpyDeviceToHost));
    CK(nullptr, cudaMemcpy(off_inout, d_off.p, sizeof(double2), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

int sdrb_host_alloc(size_t bytes, void **ptr_out)
{
    if (!ptr_out) return fail(nullptr, SDRB_ERR_ARG, "null argument");
    CK(nullptr, cudaHostAlloc(ptr_out, bytes ? bytes : 1, cudaHostAllocDefault));
    return SDRB_OK;
}

int sdrb_host_free(void *ptr)
{
    if (ptr) CK(nullptr, cudaFreeHost(ptr));
    return SDRB_OK;
}

int sdrb_keep_x0(sdrb_handle *h, int on)
{
    if (!h) return fail(h, SDRB_ERR_ARG, "null argument");
    if (!h->tc_on) return fail(h, SDRB_ERR_STATE, "block first samples exist only on the tensor-core front end");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaDeviceSynchronize());
    if (on && !h->x0_buf) {
        int rc = dalloc(h, h->max_chunks * (size_t)h->pl.R * h->pl.Mf, &h->x0_buf);
        if (rc) return rc;
    }
    h->sc.x0 = on ? h->x0_buf : nullptr;
    return SDRB_OK;
}

int sdrb_read_x0(sdrb_handle *h, size_t nchunks, double *x0_host)
{
    if (!h || !x0_host) return fail(h, SDRB_ERR_ARG, "null argument");
    if (!h->sc.x0) return fail(h, SDRB_ERR_STATE, "block first samples not kept: call sdrb_keep_x0(h, 1) first");
    if (nchunks > h->last_nchunks) return fail(h, SDRB_ERR_STATE, "only %zu chunks in the last batch", h->last_nchunks);
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(x0_host, h->sc.x0, nchunks * (size_t)h->pl.R * h->pl.Mf * sizeof(double2), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

}  // extern "C"
