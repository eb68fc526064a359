// omega4_cuda.cu -- host side of libomega4_cuda.so: the C ABI declared in include/omega4_cuda.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include "../../include/omega4_cuda.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "bars_kernel.cuh"
#include "blockdft_kernel.cuh"
#include "blockdft_tc_kernel.cuh"
#include "fft_core.cuh"
#include "kweight_kernel.cuh"
#include "kweight32_kernel.cuh"
#include "loudness_kernel.cuh"
#include "misc_kernels.cuh"
#include "octave_kernel.cuh"
#include "multires_kernel.cuh"
#include "stats_kernel.cuh"
#include "truepeak_kernel.cuh"
#include "truepeak16_kernel.cuh"
#include "waterfall_kernel.cuh"

using namespace o4;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CK(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char b__[512];                                                                         \
            snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),     \
                     __FILE__, __LINE__);                                                          \
            return fail(OMEGA4_ERR_CUDA, b__);                                                     \
        }                                                                                          \
    } while (0)

extern "C" const char* omega4_last_error(void) { return g_err.c_str(); }
extern "C" int omega4_abi_version(void) { return OMEGA4_ABI_VERSION; }
extern "C" int omega4_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static int ilog2(int n) { int l = 0; while ((1 << l) < n) ++l; return l; }
static bool is_pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }

// ------------------------------------------------------------------------------------------
// twiddle tables, cached per (device, log2M)
// ------------------------------------------------------------------------------------------
struct Twiddles { float2* twM = nullptr; float2* twN = nullptr; float2* tw4W = nullptr; };
static std::mutex g_tw_mu;
static std::map<std::pair<int, int>, Twiddles> g_tw;

static int get_twiddles(int device, int log2m, Twiddles* out) {
    std::lock_guard<std::mutex> lk(g_tw_mu);
    auto key = std::make_pair(device, log2m);
    auto it = g_tw.find(key);
    if (it != g_tw.end()) { *out = it->second; return OMEGA4_OK; }
    const int M = 1 << log2m, N = 2 * M;
    const double two_pi = 6.283185307179586476925287;
    std::vector<float2> a(M), b(M / 2 + 1), c(3 * M + 1);
    for (int e = 0; e < M; ++e) a[e] = make_float2((float)cos(two_pi * e / M), (float)-sin(two_pi * e / M));
    for (int k = 0; k <= M / 2; ++k) b[k] = make_float2((float)cos(two_pi * k / N), (float)-sin(two_pi * k / N));
    for (int j = 0; j <= 3 * M; ++j) c[j] = make_float2((float)cos(two_pi * j / (4.0 * N)), (float)sin(two_pi * j / (4.0 * N)));
    Twiddles t;
    CK(cudaMalloc(&t.twM, a.size() * sizeof(float2)));
    CK(cudaMalloc(&t.twN, b.size() * sizeof(float2)));
    CK(cudaMalloc(&t.tw4W, c.size() * sizeof(float2)));
    CK(cudaMemcpy(t.twM, a.data(), a.size() * sizeof(float2), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(t.twN, b.data(), b.size() * sizeof(float2), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(t.tw4W, c.data(), c.size() * sizeof(float2), cudaMemcpyHostToDevice));
    g_tw[key] = t;
    *out = t;
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// kernel launch dispatch over the transform size
// ------------------------------------------------------------------------------------------
template <int L>
static int launch_multires_t(const MultiresArgs& a, cudaStream_t s) {
    using S = FftShape<L>;
    const int fpc = a.rounds * S::CONC;
    const long long tiles = (a.n_frames + fpc - 1) / fpc;
    const long long grid = tiles * a.n_ch;
    if (grid <= 0) return OMEGA4_OK;
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "multires grid too large");
    if constexpr (L <= 12) {
        const size_t smem = multires_local_smem_bytes<L>(a.need_cnt, a.n_tb);
        CK(cudaFuncSetAttribute(multires_local_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        multires_local_kernel<L><<<(unsigned)grid, 256, smem, s>>>(a);
    } else {
        const size_t smem = multires_smem_bytes<L>(a.need_cnt);
        CK(cudaFuncSetAttribute(multires_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        multires_kernel<L><<<(unsigned)grid, S::NT, smem, s>>>(a);
    }
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

static int launch_multires(int log2m, const MultiresArgs& a, cudaStream_t s) {
    switch (log2m) {
        case 8: return launch_multires_t<8>(a, s);
        case 9: return launch_multires_t<9>(a, s);
        case 10: return launch_multires_t<10>(a, s);
        case 11: return launch_multires_t<11>(a, s);
        case 12: return launch_multires_t<12>(a, s);
        case 13: return launch_multires_t<13>(a, s);
        case 14: return launch_multires_t<14>(a, s);
    }
    return fail(OMEGA4_ERR_UNSUPPORTED, "fft size must be a power of two in 512 .. 32768");
}

static int default_rounds(int n_frames, int conc) {
    // enough rounds to amortise the per-thread window/twiddle loads, few enough to keep the grid large
    int r = 16;
    while (r > 1 && (long long)r * conc > n_frames) r >>= 1;
    return r;
}

static void fill_truepeak_steps(TruePeakArgs* t) {
    const double two_pi = 6.283185307179586476925287;
    for (int p = 1; p <= 3; ++p) {
        for (int j = 0; j < 16; ++j) {
            const int jj = j < 8 ? j : j - 16;
            t->step[p - 1][j] = make_float2((float)cos(two_pi * p * jj / 64.0), (float)sin(two_pi * p * jj / 64.0));
        }
        t->nyq[p - 1] = (float)cos(two_pi * p / 8.0);
    }
}

static int launch_truepeak(const TruePeakArgs& a, cudaStream_t s) {
    constexpr int L = 11;     // W = 2048 complex points: two real frames per transform
    using S = FftShape<L>;
    const size_t smem = truepeak_smem_bytes<L>();
    CK(cudaFuncSetAttribute(truepeak_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ppc = a.rounds * S::CONC;                    // frame pairs per CTA
    const int n_pairs = (a.n_frames + 1) / 2;
    const long long grid = (long long)((n_pairs + ppc - 1) / ppc) * a.n_ch;
    if (grid <= 0) return OMEGA4_OK;
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "truepeak grid too large");
    truepeak_kernel<L><<<(unsigned)grid, S::NT, smem, s>>>(a);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

static int launch_truepeak16(const TruePeakArgs& a, cudaStream_t s) {
    constexpr int L = 11;
    using S = FftShape<L>;
    const size_t smem = truepeak16_smem_bytes<L>();
    CK(cudaFuncSetAttribute(truepeak16_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ppc = a.rounds * S::CONC;                    // frame pairs per CTA
    const int n_pairs = (a.n_frames + 1) / 2;
    const long long grid = (long long)((n_pairs + ppc - 1) / ppc) * a.n_ch;
    if (grid <= 0) return OMEGA4_OK;
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "truepeak grid too large");
    truepeak16_kernel<L><<<(unsigned)grid, S::NT, smem, s>>>(a);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

template <bool F64, bool WT>
static int launch_kweight_t(const KweightArgs& a, cudaStream_t s) {
    const size_t smem = kweight_smem_bytes();
    CK(cudaFuncSetAttribute(kweight_kernel<F64, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int fpc = a.frames_per_warp * KW_WARPS;
    const long long grid = (long long)((a.n_frames + fpc - 1) / fpc) * a.n_ch;
    if (grid <= 0) return OMEGA4_OK;
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "kweight grid too large");
    kweight_kernel<F64, WT><<<(unsigned)grid, KW_WARPS * 32, smem, s>>>(a);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

static int launch_kweight(const KweightArgs& a, cudaStream_t s) {
    if (a.x_is_f64) return a.weighted_out ? launch_kweight_t<true, true>(a, s) : launch_kweight_t<true, false>(a, s);
    return a.weighted_out ? launch_kweight_t<false, true>(a, s) : launch_kweight_t<false, false>(a, s);
}

static int launch_kweight32(const Kweight32Args& a, cudaStream_t s) {
    const size_t smem = kweight32_smem_bytes();
    CK(cudaFuncSetAttribute(kweight32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int fpc = a.frames_per_warp * KW32_WARPS;
    const long long grid = (long long)((a.n_frames + fpc - 1) / fpc) * a.n_ch;
    if (grid <= 0) return OMEGA4_OK;
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "kweight grid too large");
    kweight32_kernel<<<(unsigned)grid, KW32_WARPS * 32, smem, s>>>(a);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

static int launch_stats(const StatsArgs& a, cudaStream_t s) {
    if (a.n_ch <= 0) return OMEGA4_OK;
    if (!a.fresh && a.n_frames == 1 && a.first_frame == 0 && !getenv("OMEGA4_STATS_WALK")) {
        stats_push1_kernel<<<a.n_ch, ST_P1_THREADS, 0, s>>>(a);       // one frame on carried state: block-wide sort
    } else if (a.fresh) {                            // no carried state to sort: 14.7 KB per channel, 15 channels per SM
        const size_t smem = stats_smem_bytes<false>();
        CK(cudaFuncSetAttribute(stats_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        stats_kernel<false><<<a.n_ch, ST_THREADS, smem, s>>>(a);
    } else {
        const size_t smem = stats_smem_bytes<true>();
        CK(cudaFuncSetAttribute(stats_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        stats_kernel<true><<<a.n_ch, ST_THREADS, smem, s>>>(a);
    }
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

static int launch_s16_convert(const int16_t* in, long long stream_stride, int il, int n_streams, long long n_frames,
                              float* out, long long out_stride, cudaStream_t s) {
    if (n_streams <= 0 || n_frames <= 0) return OMEGA4_OK;
    if (n_streams > 65535) return fail(OMEGA4_ERR_INVALID, "too many streams for one int16 conversion launch (max 65535)");
    const long long per_stream = n_frames * il;
    dim3 grid((unsigned)((per_stream + 1023) / 1024), (unsigned)n_streams);
    s16_deinterleave_kernel<<<grid, 256, 0, s>>>(in, stream_stride, il, n_frames, out, out_stride);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// K-weighting scan tables
// ------------------------------------------------------------------------------------------
static void mat2_mul(const double* a, const double* b, double* c) {
    double r[4] = {a[0] * b[0] + a[1] * b[2], a[0] * b[1] + a[1] * b[3],
                   a[2] * b[0] + a[3] * b[2], a[2] * b[1] + a[3] * b[3]};
    memcpy(c, r, sizeof r);
}

// b, a: order + 1 coefficients (order 1 or 2).  Everything the scan needs is derived here in float64.
static void build_biquad(const double* b, const double* a, int order, KwBiquad* q) {
    memset(q, 0, sizeof *q);
    const double a0 = a[0];
    q->b0 = b[0] / a0; q->b1 = b[1] / a0; q->b2 = order >= 2 ? b[2] / a0 : 0.0;
    q->a1 = a[1] / a0; q->a2 = order >= 2 ? a[2] / a0 : 0.0;
    q->pad = 3 * (order + 1);                                // scipy filtfilt default padlen
    if (order >= 2) {
        // lfilter_zi: (I - companion(a)^T) zi = b[1:] - a[1:] b[0]
        double zi0, zi1;
        const double m00 = 1.0 + q->a1, m01 = -1.0, m10 = q->a2, m11 = 1.0;
        const double r0 = q->b1 - q->a1 * q->b0, r1 = q->b2 - q->a2 * q->b0;
        const double det = m00 * m11 - m01 * m10;
        zi0 = (r0 * m11 - m01 * r1) / det;
        zi1 = (m00 * r1 - m10 * r0) / det;
        // direct form I initial outputs equivalent to the transposed-form-II state (zi0, zi1) with
        // x[-1] = x[-2] = 0:  -a1 y[-1] - a2 y[-2] = zi0,  -a2 y[-1] = zi1
        q->yi0 = -zi1 / q->a2;
        q->yi1 = (-zi0 + q->a1 * zi1 / q->a2) / q->a2;
    } else {
        // first order: zi = (b1 - a1 b0) / (1 + a1);  -a1 y[-1] = zi
        const double zi0 = (q->b1 - q->a1 * q->b0) / (1.0 + q->a1);
        q->yi0 = -zi0 / q->a1;
        q->yi1 = 0.0;
    }
    // companion matrix of the output recursion: (y[n], y[n-1]) = C (y[n-1], y[n-2])
    const double Cm[4] = {-q->a1, -q->a2, 1.0, 0.0};
    double P[4] = {Cm[0], Cm[1], Cm[2], Cm[3]};       // C^(i+1)
    for (int i = 0; i < KW_L; ++i) {
        if (i < KW_SUBMAX) { q->g[i][0] = P[0]; q->g[i][1] = P[1]; }
        if (i + 1 == 16) memcpy(q->c16, P, sizeof P);
        if (i + 1 == 17) memcpy(q->c17, P, sizeof P);
        if (i + 1 < KW_L) mat2_mul(Cm, P, P);
    }
    memcpy(q->phi[0], P, sizeof P);              // C^65
    for (int j = 1; j < 5; ++j) mat2_mul(q->phi[j - 1], q->phi[j - 1], q->phi[j]);
    // C^-k for the two virtual start offsets
    auto inv_pow = [&](int k, double* out) {
        if (k == 0) { out[0] = 1; out[1] = 0; out[2] = 0; out[3] = 1; return; }
        if (order >= 2) {
            const double det1 = Cm[0] * Cm[3] - Cm[1] * Cm[2];           // = a2
            const double Ci[4] = {Cm[3] / det1, -Cm[1] / det1, -Cm[2] / det1, Cm[0] / det1};
            double R[4] = {Ci[0], Ci[1], Ci[2], Ci[3]};
            for (int i = 1; i < k; ++i) mat2_mul(Ci, R, R);
            memcpy(out, R, sizeof R);
        } else {                                                       // singular companion: scalar recursion
            out[0] = pow(-q->a1, -(double)k); out[1] = 0; out[2] = 0; out[3] = 0;
        }
    };
    inv_pow(KW_PAD - q->pad, q->cinv_f);
    inv_pow(KW_SLACK + KW_PAD - q->pad, q->cinv_b);
}

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
struct ResInfo {
    int n = 0, log2m = 0, bins = 0;
    float weight = 1.f;
    float* window = nullptr;
    float* binw = nullptr;
    int n_tb = 0;                 // entries in the device tables (incl. orphans on resolution 0)
    int* tb_idx = nullptr;
    int* tb_lo = nullptr;
    float* tb_frac = nullptr;
    int need_lo = 0, need_cnt = 0;
    Twiddles tw;
};

// A resolution whose fused output needs only a few FFT bins (blockdft_kernel.cuh)
struct SparseRes {
    int r = 0, nk = 0, nt = 0, B = 0, col0 = 0;
    bool td = false;              // time-domain windowed operand: one column pair per (bin, block position), no T
    int xoff = 0;                 // first bin of this resolution in the fused X rows
    float2* T = nullptr;          // [nk][B][nt]
    float* kw = nullptr;          // [nk]
    int* tb_pos = nullptr;        // [n_tb]
};

// The resolutions one GEMM over the hop blocks serves, and its constant operand
struct SparseSet {
    int n = 0;
    SparseRes sp[OMEGA4_MAX_RES];
    int of_res[OMEGA4_MAX_RES];   // index into sp for resolution r, or -1
    int cols = 0, qs = 0;         // used GEMM columns, Q row stride (padded columns)
    float* E = nullptr;           // CUDA-core GEMM operand [hop][qs]            (blockdft_kernel.cuh)
    uint8_t* Eimg = nullptr;      // tensor-core operand images, hi/lo, swizzled  (blockdft_tc_kernel.cuh)
    float e_inv = 1.f;            // inverse of the images' power-of-two scale (half operands)
    int n_halves = 0;
    // fused frame assembly in the GEMM epilogue: possible when every resolution of the set uses the exact-
    // windowing operand with 2 / 4 / 8 / 16 block positions per bin and 32-column aligned blocks
    bool fusable = false;
    int nkx = 0;                  // bins per frame over all resolutions of the set
    short gB[TC_MAX_GROUPS], gX[TC_MAX_GROUPS], gN[TC_MAX_GROUPS], gS[TC_MAX_GROUPS]; // per 32-column group of the GEMM: positions per bin, first bin, bins present, frame shift
    SparseSet() { for (int i = 0; i < OMEGA4_MAX_RES; ++i) of_res[i] = -1; }
    void release() {
        for (int i = 0; i < OMEGA4_MAX_RES; ++i) { cudaFree(sp[i].T); cudaFree(sp[i].kw); cudaFree(sp[i].tb_pos); }
        cudaFree(E); cudaFree(Eimg);
    }
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return OMEGA4_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        CK(cudaMalloc(&p, bytes));
        cap = bytes;
        return OMEGA4_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// ------------------------------------------------------------------------------------------
// application post-processing object (omega4_bars_*); also used fused behind the combine by omega4_analyze_io
// ------------------------------------------------------------------------------------------
struct omega4_bars {
    int device = 0, T = 0, n_valid = 0, p_lo = 0, normalize_max = 0;
    float p_frac = 0.f, scale = 0.8f;
    int* bands = nullptr; float* gain = nullptr; float* sf = nullptr; float* sfc = nullptr;
    DevBuf h_spec, h_out, h_peak, h_state, state_in;
};

// spectrum [n_ch][n_hops][T] (device) -> band values (+ unsmoothed peaks) on stream s; state (device) carries the
// smoothing recurrence between calls.  state_copy: scratch for the private copy segment 0 reads when a channel is cut
// into several segments (the last segment overwrites the state in the same launch).
static int bars_launch(omega4_bars* b, cudaStream_t s, const float* spec, int n_ch, int n_hops, float* state, int fresh,
                       float* band_values, float* peak_values, DevBuf* state_copy) {
    BarsArgs a;
    memset(&a, 0, sizeof a);
    a.T = b->T; a.n_ch = n_ch; a.n_hops = n_hops; a.n_valid = b->n_valid; a.bands = b->bands; a.gain = b->gain;
    a.sf = b->sf; a.sfc = b->sfc; a.p_lo = b->p_lo; a.p_frac = b->p_frac; a.scale = b->scale;
    a.normalize_max = b->normalize_max; a.fresh = (fresh || !state) ? 1 : 0;
    a.spec = spec; a.bars_out = band_values; a.peaks_out = peak_values; a.state = state;
    const size_t st_bytes = (size_t)n_ch * (1 + b->n_valid) * sizeof(float);
    const size_t smem = bars_smem_bytes(b->T, b->n_valid);
    if (smem > 200 * 1024) return fail(OMEGA4_ERR_UNSUPPORTED, "spectrum too long for the bars kernel");
    if (b->T > 32 * BARS_MAXV) return fail(OMEGA4_ERR_UNSUPPORTED, "spectrum too long for the bars kernel (max 1024 bins)");
    if (b->T <= 512) CK(cudaFuncSetAttribute(bars_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    else CK(cudaFuncSetAttribute(bars_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    a.seg = n_ch >= 1024 ? 4 * BARS_SEG : BARS_SEG;              // fewer warm-up replays when channels alone fill the GPU
    const long long grid = (long long)n_ch * ((n_hops + a.seg - 1) / a.seg);
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "bars grid too large");
    if (a.state && !a.fresh && n_hops > a.seg) {
        int rc = state_copy->ensure(st_bytes); if (rc) return rc;
        CK(cudaMemcpyAsync(state_copy->p, a.state, st_bytes, cudaMemcpyDeviceToDevice, s));
        a.state_in = (const float*)state_copy->p;
    }
    if (b->T <= 512) bars_kernel<16><<<(unsigned)grid, BARS_WARPS * 32, smem, s>>>(a);
    else bars_kernel<32><<<(unsigned)grid, BARS_WARPS * 32, smem, s>>>(a);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

// what omega4_analyze_io adds to a plain analyze call
struct BarsReq {
    omega4_bars* b = nullptr;
    float* band_values = nullptr; float* peak_values = nullptr; float* state = nullptr;
    int fresh = 1;
};

struct KernelTime { char name[32]; cudaEvent_t e0, e1; };

// side stream + fork/join events of one caller stream (plan-level for device calls, one per host slot)
struct SideCtx {
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_tp = nullptr, ev_join = nullptr;
    int ensure() {
        if (side) return OMEGA4_OK;
        CK(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_tp, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        return OMEGA4_OK;
    }
    void release() {
        if (side) cudaStreamDestroy(side);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_tp) cudaEventDestroy(ev_tp);
        if (ev_join) cudaEventDestroy(ev_join);
        side = nullptr; ev_fork = ev_tp = ev_join = nullptr;
    }
};

struct omega4_plan {
    int device = 0;
    int sample_rate = 48000, hop = 512, n_res = 0, T = 0, W = OMEGA4_METER_WINDOW;
    double gate = -70.0;
    ResInfo res[OMEGA4_MAX_RES];
    bool disjoint = true;
    // general combine CSR
    int* csr_ptr = nullptr; int* csr_res = nullptr; int* csr_lo = nullptr; float* csr_frac = nullptr;
    double* hann64 = nullptr;
    float* hann32 = nullptr;
    KwBiquad kw_default[2];       // the K-weighting pair of the plan descriptor
    KwBiquad kw[4];               // active weighting program (omega4_plan_set_weighting)
    int kw_nsec = 2, kw_blend = 1, kw_gate = 1;
    double kw_gain = 1.0;
    Twiddles tw_meter;            // W-point complex transform of the true-peak kernel
    float2* tp_rot = nullptr;     // [3][W] fractional-delay factors
    unsigned* tp_rot_h = nullptr; // the same as packed half (re, im) for the all-half kernel
    SparseSet set_cc;             // fp32 CUDA-core GEMM: up to 128 columns
    SparseSet set_tc;             // 3xTF32 tcgen05 GEMM: up to 512 columns
    bool tensor_default = true;   // OMEGA4_TENSOR=0 makes the CUDA-core GEMM the default
    DevBuf scratch_lufs, scratch_tp, scratch_mag[OMEGA4_MAX_RES], scratch_q, scratch_f32, scratch_comb, scratch_bstate, scratch_inv;
    DevBuf h_in, h_comb, h_meters, h_state, h_mag[OMEGA4_MAX_RES], h_f64a, h_f64b, h_f64c;
    // host-buffer mode: channel chunks are pipelined over N_SLOTS private streams / buffer sets so
    // that H2D of chunk i+1, the kernels of chunk i and D2H of chunk i-1 overlap
    struct Slot {
        cudaStream_t s = nullptr;
        DevBuf in, in16, comb, met, lufs, tp, state, q, mag[OMEGA4_MAX_RES];
        DevBuf bars, peaks, bstate, bstate_copy;          // omega4_analyze_io: fused application post-processing
        SideCtx sc;
    };
#ifndef OMEGA4_HOST_SLOTS
#define OMEGA4_HOST_SLOTS 4
#endif
    static constexpr int N_SLOTS = OMEGA4_HOST_SLOTS;
    Slot slots[N_SLOTS];
    size_t host_chunk_bytes = (size_t)1024 << 20;  // device bytes per slot (OMEGA4_HOST_CHUNK_MB overrides)
    // OMEGA4_FLAG_CONCURRENT_METERS: the K-weighting + stats kernels run on a side stream, forked /
    // joined with events on the caller's stream
    SideCtx sc;
    long long launches = 0;
    std::vector<KernelTime> times;
    size_t n_times = 0;
};

static void set_weighting_k(omega4_plan* p) {
    p->kw[0] = p->kw_default[0]; p->kw[1] = p->kw_default[1];
    p->kw_nsec = 2; p->kw_blend = 1; p->kw_gate = 1; p->kw_gain = 1.0;
}

static double max_pole_radius(const KwBiquad& q) {
    if (q.a2 == 0.0) return fabs(q.a1);
    const double disc = q.a1 * q.a1 - 4.0 * q.a2;
    if (disc < 0.0) return sqrt(q.a2);
    return fmax(fabs(-q.a1 + sqrt(disc)), fabs(-q.a1 - sqrt(disc))) * 0.5;
}

static void to_float(const KwBiquad& s, KwBiquadF* d) {
    d->b0 = (float)s.b0; d->b1 = (float)s.b1; d->b2 = (float)s.b2; d->a1 = (float)s.a1; d->a2 = (float)s.a2;
    d->yi0 = (float)s.yi0; d->yi1 = (float)s.yi1; d->pad = s.pad; d->_align = 0;
    for (int j = 0; j < 5; ++j) for (int e = 0; e < 4; ++e) d->phi[j][e] = (float)s.phi[j][e];
    for (int e = 0; e < 4; ++e) {
        d->cinv_f[e] = (float)s.cinv_f[e]; d->cinv_b[e] = (float)s.cinv_b[e];
        d->c16[e] = (float)s.c16[e]; d->c17[e] = (float)s.c17[e];
    }
    for (int i = 0; i < KW_SUBMAX; ++i) { d->g[i][0] = (float)s.g[i][0]; d->g[i][1] = (float)s.g[i][1]; }
}

// float32-state form of one high-pass section (kweight32_kernel.cuh): b = b0 [1, -2, 1] required
static bool is_highpass_biquad(const KwBiquad& q) {
    return q.pad == 9 && q.a2 != 0.0 && fabs(q.b1 + 2.0 * q.b0) <= 1e-12 * fabs(q.b0) && fabs(q.b2 - q.b0) <= 1e-12 * fabs(q.b0);
}

static void build_kw32(const KwBiquad& q, Kw32Sec* o) {
    const double alpha = 1.0 + q.a1 + q.a2, beta = 1.0 - q.a2;
    const double bb = -q.b0 * beta, gamma = alpha / bb;
    o->b0 = (float)q.b0; o->a2 = (float)q.a2; o->gamma = (float)gamma; o->bb = (float)bb;
    const double M[4] = {1.0 - alpha, bb * q.a2, -gamma, q.a2}; // (z, delta) -> (z + bb delta', delta'),  delta' = a2 delta - gamma z
    double P[4] = {M[0], M[1], M[2], M[3]};
    for (int i = 0; i < KW_L; ++i) {                            // P = M^(i+1)
        if (i < KW_SUBMAX) { o->g[i][0] = (float)P[0]; o->g[i][1] = (float)P[1]; }
        if (i + 1 == 16) for (int e = 0; e < 4; ++e) o->c16[e] = (float)P[e];
        if (i + 1 == 17) for (int e = 0; e < 4; ++e) o->c17[e] = (float)P[e];
        if (i + 1 < KW_L) mat2_mul(M, P, P);
    }
    for (int k = 0; k < 16; ++k) {
        o->ga0[k] = make_float2(o->g[k + 1][0], o->g[k][0]);
        o->ga1[k] = make_float2(o->g[k + 1][1], o->g[k][1]);
    }
    double Q[4] = {P[0], P[1], P[2], P[3]};                     // M^65
    for (int j = 0; j < 5; ++j) {
        for (int e = 0; e < 4; ++e) o->phi[j][e] = (float)Q[e];
        mat2_mul(Q, Q, Q);
    }
}

// the batch path's K-weighting runs in the float32-state kernel when the active program is the two
// high-pass sections blended as f + 0.3 (s - f) (the default); OMEGA4_KW_F64=1 keeps the float64 kernel
static bool use_kweight32(const omega4_plan* p) {
    return p->W == KW_W && p->kw_nsec == 2 && p->kw_blend && p->kw_gain == 1.0 && is_highpass_biquad(p->kw[0]) &&
           is_highpass_biquad(p->kw[1]) && !getenv("OMEGA4_KW_F64");
}

static void fill_weighting(const omega4_plan* p, KweightArgs* k) {
    k->n_sec = p->kw_nsec; k->blend = p->kw_blend; k->rms_gate = p->kw_gate; k->gain = p->kw_gain;
    for (int i = 0; i < p->kw_nsec; ++i) { k->f[i] = p->kw[i]; to_float(p->kw[i], &k->ff[i]); }
    // trailing sections whose poles stay inside |z| < 0.95 run in float32 (kweight_kernel.cuh); the first
    // section always keeps float64 state
    int from = p->kw_nsec;
    while (from > 1 && max_pole_radius(p->kw[from - 1]) < 0.95) --from;
    k->f32_from = getenv("OMEGA4_KW_F64") ? p->kw_nsec : from;
}

static int upload(void** dst, const void* src, size_t bytes) {
    CK(cudaMalloc(dst, bytes ? bytes : 1));
    if (bytes) CK(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return OMEGA4_OK;
}

static size_t boff_of(const omega4_plan_desc* d, int r) {
    size_t o = 0;
    for (int i = 0; i < r; ++i) o += (size_t)d->fft_sizes[i] / 2 + 1;
    return o;
}

// ------------------------------------------------------------------------------------------
// hop-block partial DFT tables (blockdft_kernel.cuh / blockdft_tc_kernel.cuh)
// ------------------------------------------------------------------------------------------
static int build_sparse_set(omega4_plan* p, const omega4_plan_desc* d, const std::vector<std::vector<int>>& idx,
                            const std::vector<std::vector<int>>& lo, bool tensor, SparseSet* set) {
    const int H = d->hop;
    if ((H % (tensor ? TC_KC : BD_KC)) != 0) return OMEGA4_OK;
    // tensor: up to eight column tiles of 256 (each tile = all 512 TMEM columns as main | cross; config 5 fits its 32768,
    // 16384 and 8192-point transforms in 256 + 512 + 1280 = 2048 columns); CUDA cores: the widest tile
    const int max_cols = tensor ? TC_MAX_GROUPS * 32 : 128;
    // exact (time-domain) windowing for the tensor-core set: one column pair per (bin, block position), up to 64
    // hop blocks per frame (config 5: 32768 / 16384 at hop 512 take 2 x 2 x 64 + 2 x 8 x 32 = 768 columns).  The
    // cosine-sum formulation loses up to 0.03 dB on a click under the window's near-zero edge (DESIGN.md 4.1b) and
    // is only built on request: OMEGA4_BLOCKDFT_FD=1 forces it everywhere.
    const bool allow_td = tensor && !getenv("OMEGA4_BLOCKDFT_FD");
    int order[OMEGA4_MAX_RES];
    for (int r = 0; r < d->n_res; ++r) order[r] = r;
    for (int i = 0; i < d->n_res; ++i)                 // largest transform first
        for (int j = i + 1; j < d->n_res; ++j)
            if (p->res[order[j]].n > p->res[order[i]].n) { int t = order[i]; order[i] = order[j]; order[j] = t; }
    std::vector<std::vector<float>> ecols;             // per accepted resolution: [hop][2 nk nt]
    int cols = 0;
    size_t woff2[OMEGA4_MAX_RES];
    { size_t o = 0; for (int r = 0; r < d->n_res; ++r) { woff2[r] = o; o += d->fft_sizes[r]; } }
    for (int oi = 0; oi < d->n_res; ++oi) {
        const int r = order[oi];
        const ResInfo& ri = p->res[r];
        const int N = ri.n;
        if (N % H != 0 || N / H < 2 || N / H > 64) continue;
        std::vector<int> bins;
        for (int l : lo[r]) if (l >= 0) { bins.push_back(l); bins.push_back(l + 1); }
        std::sort(bins.begin(), bins.end());
        bins.erase(std::unique(bins.begin(), bins.end()), bins.end());
        if (bins.empty()) continue;
        const float* w = d->windows + woff2[r];
        const double two_pi = 6.283185307179586476925287;
        const int nk = (int)bins.size();
        const double fft_cost = 2.5 * N * (ri.log2m + 1);
        if (allow_td && N / H <= 64 && (double)(2 * nk * (N / H)) * H <= 6.6 * fft_cost &&
            ((cols + 31) & ~31) + 2 * nk * (N / H) <= max_cols) {
            // ---- exact windowing: column pair (ki, b) = w[H b + n] e^{-2 pi i k (H b + n) / N}
            cols = (cols + 31) & ~31;                      // whole 32-column groups per resolution (fused epilogue)
            SparseRes& sp = set->sp[set->n];
            sp.r = r; sp.nk = nk; sp.nt = N / H; sp.B = N / H; sp.col0 = cols; sp.td = true;
            const int rc_cols = 2 * nk * sp.B;
            std::vector<float> ec((size_t)H * rc_cols);
            std::vector<float> kw(nk);
            for (int ki = 0; ki < nk; ++ki) {
                kw[ki] = d->bin_weights ? d->bin_weights[boff_of(d, r) + bins[ki]] : 1.f;
                for (int b = 0; b < sp.B; ++b)
                    for (int n2 = 0; n2 < H; ++n2) {
                        const int i = H * b + n2;
                        const long long ph = ((long long)bins[ki] * i) % N;              // exact phase reduction
                        const double ang = -two_pi * (double)ph / (double)N;
                        ec[(size_t)n2 * rc_cols + 2 * (ki * sp.B + b)] = (float)((double)w[i] * cos(ang));
                        ec[(size_t)n2 * rc_cols + 2 * (ki * sp.B + b) + 1] = (float)((double)w[i] * sin(ang));
                    }
            }
            std::vector<int> pos(idx[r].size(), -1);
            for (size_t j = 0; j < lo[r].size(); ++j)
                if (lo[r][j] >= 0) pos[j] = (int)(std::lower_bound(bins.begin(), bins.end(), lo[r][j]) - bins.begin());
            int rc = upload((void**)&sp.kw, kw.data(), kw.size() * sizeof(float)); if (rc) return rc;
            rc = upload((void**)&sp.tb_pos, pos.data(), pos.size() * sizeof(int)); if (rc) return rc;
            set->of_res[r] = set->n++;
            ecols.push_back(std::move(ec));
            cols += rc_cols;
            cols = (cols + 31) & ~31;
            continue;
        }
        // least-squares fit  w[i] = a0 + a1 cos(phi i) + a2 cos(2 phi i),  phi = 2 pi / (N - 1)
        const double phi = 6.283185307179586476925287 / (double)(N - 1);
        double G[3][4] = {{0}};
        for (int i = 0; i < N; ++i) {
            const double c[3] = {1.0, cos(phi * i), cos(2.0 * phi * i)};
            for (int u = 0; u < 3; ++u) { for (int v = 0; v < 3; ++v) G[u][v] += c[u] * c[v]; G[u][3] += c[u] * (double)w[i]; }
        }
        bool singular = false;
        for (int u = 0; u < 3 && !singular; ++u) {        // Gauss-Jordan with partial pivoting
            int piv = u;
            for (int v = u + 1; v < 3; ++v) if (fabs(G[v][u]) > fabs(G[piv][u])) piv = v;
            if (fabs(G[piv][u]) < 1e-9) { singular = true; break; }
            if (piv != u) for (int c2 = 0; c2 < 4; ++c2) { double t = G[u][c2]; G[u][c2] = G[piv][c2]; G[piv][c2] = t; }
            for (int v = 0; v < 3; ++v) {
                if (v == u) continue;
                const double f = G[v][u] / G[u][u];
                for (int c2 = 0; c2 < 4; ++c2) G[v][c2] -= f * G[u][c2];
            }
        }
        if (singular) continue;
        double am[3] = {G[0][3] / G[0][0], G[1][3] / G[1][1], G[2][3] / G[2][2]};
        double resid = 0.0;
        for (int i = 0; i < N; ++i) {
            const double fit = am[0] + am[1] * cos(phi * i) + am[2] * cos(2.0 * phi * i);
            resid = fmax(resid, fabs(fit - (double)w[i]));
        }
        if (resid > 1.5e-7) continue;                     // not a cosine-sum window: keep the FFT path
        int tm[5]; double tc[5]; int nt = 0;
        tm[nt] = 0; tc[nt] = am[0]; ++nt;
        for (int m = 1; m <= 2; ++m)
            if (fabs(am[m]) > 1e-9) { tm[nt] = m; tc[nt] = 0.5 * am[m]; ++nt; tm[nt] = -m; tc[nt] = 0.5 * am[m]; ++nt; }
        const int rc_cols = 2 * nk * nt;
        // cost model against the FFT kernel's ~2.5 N log2 N instructions per frame (measured ~22 T instr/s):
        //   CUDA-core GEMM: cols x hop FMAs at ~23 T/s  -> accept below half the FFT's count
        //   tensor-core GEMM: 3 x cols x hop MACs at ~250 T/s (measured, 3xTF32)
        if (!tensor && (double)rc_cols * H * 2.0 > fft_cost) continue;
        if (tensor && (double)rc_cols * H > 6.6 * fft_cost) continue;
        if (cols + rc_cols > max_cols) continue;
        SparseRes& sp = set->sp[set->n];
        sp.r = r; sp.nk = nk; sp.nt = nt; sp.B = N / H; sp.col0 = cols;
        std::vector<float> ec((size_t)H * rc_cols);
        std::vector<float2> T((size_t)nk * sp.B * nt);
        std::vector<float> kw(nk);
        for (int ki = 0; ki < nk; ++ki) {
            kw[ki] = d->bin_weights ? d->bin_weights[boff_of(d, r) + bins[ki]] : 1.f;
            for (int t = 0; t < nt; ++t) {
                const double th = tm[t] * phi - two_pi * (double)bins[ki] / (double)N;
                for (int n2 = 0; n2 < H; ++n2) {
                    const double ang = fmod(th * n2, two_pi);
                    ec[(size_t)n2 * rc_cols + 2 * (ki * nt + t)] = (float)cos(ang);
                    ec[(size_t)n2 * rc_cols + 2 * (ki * nt + t) + 1] = (float)sin(ang);
                }
                for (int b = 0; b < sp.B; ++b) {
                    const double ang = fmod(th * (double)H * b, two_pi);
                    T[((size_t)ki * sp.B + b) * nt + t] = make_float2((float)(tc[t] * cos(ang)), (float)(tc[t] * sin(ang)));
                }
            }
        }
        std::vector<int> pos(idx[r].size(), -1);
        for (size_t j = 0; j < lo[r].size(); ++j)
            if (lo[r][j] >= 0) pos[j] = (int)(std::lower_bound(bins.begin(), bins.end(), lo[r][j]) - bins.begin());
        int rc = upload((void**)&sp.T, T.data(), T.size() * sizeof(float2)); if (rc) return rc;
        rc = upload((void**)&sp.kw, kw.data(), kw.size() * sizeof(float)); if (rc) return rc;
        rc = upload((void**)&sp.tb_pos, pos.data(), pos.size() * sizeof(int)); if (rc) return rc;
        set->of_res[r] = set->n++;
        ecols.push_back(std::move(ec));
        cols += rc_cols;
    }
    if (set->n == 0) return OMEGA4_OK;
    set->cols = cols;
    if (!tensor) {
        set->qs = cols <= 32 ? 32 : (cols <= 64 ? 64 : 128);
        std::vector<float> E((size_t)H * set->qs, 0.f);
        for (int si = 0; si < set->n; ++si) {
            const SparseRes& sp = set->sp[si];
            const int rc_cols = 2 * sp.nk * sp.nt;
            for (int n2 = 0; n2 < H; ++n2)
                memcpy(&E[(size_t)n2 * set->qs + sp.col0], &ecols[si][(size_t)n2 * rc_cols], rc_cols * sizeof(float));
        }
        return upload((void**)&set->E, E.data(), E.size() * sizeof(float));
    }
    // tensor-core operand: per column half and K chunk, the (hi, lo) TF32 split of E^T as byte images of
    // the K-major SWIZZLE_64B shared-memory layout
    set->n_halves = (cols + TC_BN - 1) / TC_BN;
    set->qs = set->n_halves * TC_BN;
    {
        bool ok = set->n_halves * (TC_BN / 32) <= TC_MAX_GROUPS;
        int xo = 0;
        for (int si = 0; si < set->n; ++si) {
            SparseRes& sp = set->sp[si];
            ok = ok && sp.td && (sp.B == 2 || sp.B == 4 || sp.B == 8 || sp.B == 16 || sp.B == 32 || sp.B == 64) && (sp.col0 % 32) == 0;
            sp.xoff = xo; xo += sp.nk;
        }
        set->nkx = xo;
        for (int g = 0; g < TC_MAX_GROUPS; ++g) { set->gB[g] = 0; set->gX[g] = 0; set->gN[g] = 0; set->gS[g] = -1; }
        if (ok)
            for (int si = 0; si < set->n; ++si) {
                const SparseRes& sp = set->sp[si];
                if (sp.B > 16) {                           // a bin spans B / 16 groups of 16 block positions each
                    const int parts = sp.B / 16;
                    for (int k0 = 0; k0 < sp.nk; ++k0)
                        for (int pt = 0; pt < parts; ++pt) {
                            const int g = (sp.col0 + 2 * (k0 * sp.B + 16 * pt)) / 32;
                            set->gB[g] = 16; set->gX[g] = (short)(sp.xoff + k0); set->gN[g] = 1;
                            set->gS[g] = (short)(sp.B - 16 * (pt + 1));
                        }
                    continue;
                }
                const int per = 16 / sp.B;                 // bins per 32-column group
                for (int k0 = 0; k0 < sp.nk; k0 += per) {
                    const int g = (sp.col0 + 2 * k0 * sp.B) / 32;
                    set->gB[g] = (short)sp.B; set->gX[g] = (short)(sp.xoff + k0);
                    set->gN[g] = (short)((sp.nk - k0 < per) ? sp.nk - k0 : per);
                }
            }
        set->fusable = ok && !getenv("OMEGA4_BLOCKDFT_UNFUSED");
    }
    const int nkc = H / TC_KC;
    std::vector<uint8_t> img((size_t)set->n_halves * nkc * 2 * TC_B_BYTES, 0);
#if TC_F16
    // one power-of-two scale for the whole table: its largest entry lands in [0.5, 1) of half's range
    float emax = 0.f;
    for (const auto& ec : ecols) for (float v : ec) emax = fmaxf(emax, fabsf(v));
    int eexp = 0;
    if (emax > 0.f) frexpf(emax, &eexp);                   // emax = [0.5, 1) 2^eexp
    const float escale = ldexpf(1.f, -eexp);
    set->e_inv = ldexpf(1.f, eexp);
#endif
    for (int si = 0; si < set->n; ++si) {
        const SparseRes& sp = set->sp[si];
        const int rc_cols = 2 * sp.nk * sp.nt;
        for (int cc = 0; cc < rc_cols; ++cc) {
            const int col = sp.col0 + cc, h = col / TC_BN, n = col % TC_BN;
            for (int k = 0; k < H; ++k) {
                const float v = ecols[si][(size_t)k * rc_cols + cc];
#if TC_F16
                const float vs = v * escale;
                const __half hh = __float2half_rn(vs);
                const __half hl = __float2half_rn((vs - __half2float(hh)) * TC_LO_SCALE);
                const int kc = k / TC_KC, e = k % TC_KC;
                const size_t base = ((size_t)(h * nkc + kc) * 2) * TC_B_BYTES;
                const int off = tc_sw64_offset(n, e >> 3) + (e & 7) * 2;
                memcpy(&img[base + off], &hh, 2);
                memcpy(&img[base + TC_B_BYTES + off], &hl, 2);
#else
                uint32_t bits; memcpy(&bits, &v, 4); bits &= 0xFFFFE000u;
                float hi; memcpy(&hi, &bits, 4);
                const float lo2 = v - hi;
                const int kc = k / TC_KC, e = k % TC_KC;
                const size_t base = ((size_t)(h * nkc + kc) * 2) * TC_B_BYTES;
                const int off = tc_sw64_offset(n, e >> 2) + (e & 3) * 4;
                memcpy(&img[base + off], &hi, 4);
                memcpy(&img[base + TC_B_BYTES + off], &lo2, 4);
#endif
            }
        }
    }
    return upload((void**)&set->Eimg, img.data(), img.size());
}

static int plan_build(omega4_plan* p, const omega4_plan_desc* d) {
    if (d->n_res < 1 || d->n_res > OMEGA4_MAX_RES) return fail(OMEGA4_ERR_INVALID, "n_res must be 1..8");
    if (d->hop <= 0 || (d->hop % 4) != 0) return fail(OMEGA4_ERR_INVALID, "hop must be a positive multiple of 4");
    if (d->target_bins < 1) return fail(OMEGA4_ERR_INVALID, "target_bins must be >= 1");
    if (d->meter_window != OMEGA4_METER_WINDOW) return fail(OMEGA4_ERR_UNSUPPORTED, "meter_window must be 2048");
    if (!d->fft_sizes || !d->windows || !d->tb_count || !d->res_weight || !d->meter_hann || !d->kw_coeffs)
        return fail(OMEGA4_ERR_INVALID, "plan_desc has NULL tables");
    p->sample_rate = d->sample_rate; p->hop = d->hop; p->n_res = d->n_res; p->T = d->target_bins;
    p->gate = d->gate_threshold;
    std::vector<int> owners(d->target_bins, 0);
    size_t woff = 0, boff = 0, toff = 0;
    std::vector<std::vector<int>> idx(d->n_res), lo(d->n_res);
    std::vector<std::vector<float>> fr(d->n_res);
    for (int r = 0; r < d->n_res; ++r) {
        ResInfo& ri = p->res[r];
        const int n = d->fft_sizes[r];
        if (!is_pow2(n) || n < 512 || n > 32768) return fail(OMEGA4_ERR_UNSUPPORTED, "fft size must be a power of two in 512 .. 32768");
        ri.n = n; ri.log2m = ilog2(n) - 1; ri.bins = n / 2 + 1; ri.weight = d->res_weight[r];
        if (ri.weight <= 0.f) return fail(OMEGA4_ERR_INVALID, "resolution weight must be positive");
        int rc = upload((void**)&ri.window, d->windows + woff, (size_t)n * sizeof(float));
        if (rc) return rc;
        if (d->bin_weights) { rc = upload((void**)&ri.binw, d->bin_weights + boff, (size_t)ri.bins * sizeof(float)); if (rc) return rc; }
        woff += n; boff += ri.bins;
        const int cnt = d->tb_count[r];
        if (cnt < 0) return fail(OMEGA4_ERR_INVALID, "negative tb_count");
        for (int j = 0; j < cnt; ++j) {
            const int ti = d->tb_idx[toff + j], l = d->tb_lo[toff + j];
            if (ti < 0 || ti >= d->target_bins || l < 0 || l + 1 >= ri.bins)
                return fail(OMEGA4_ERR_INVALID, "combine table entry out of range");
            idx[r].push_back(ti); lo[r].push_back(l); fr[r].push_back(d->tb_frac[toff + j]);
            owners[ti]++;
        }
        toff += cnt;
        rc = get_twiddles(p->device, ri.log2m, &ri.tw);
        if (rc) return rc;
    }
    p->disjoint = true;
    for (int t = 0; t < d->target_bins; ++t) if (owners[t] > 1) p->disjoint = false;
    // CSR for the general combine kernel (entries in resolution order, as `results` is iterated)
    {
        std::vector<int> ptr(d->target_bins + 1, 0), cres, clo;
        std::vector<float> cfr;
        for (int t = 0; t < d->target_bins; ++t) {
            for (int r = 0; r < d->n_res; ++r)
                for (size_t j = 0; j < idx[r].size(); ++j)
                    if (idx[r][j] == t) { cres.push_back(r); clo.push_back(lo[r][j]); cfr.push_back(fr[r][j]); }
            ptr[t + 1] = (int)cres.size();
        }
        int rc = upload((void**)&p->csr_ptr, ptr.data(), ptr.size() * sizeof(int)); if (rc) return rc;
        rc = upload((void**)&p->csr_res, cres.data(), cres.size() * sizeof(int)); if (rc) return rc;
        rc = upload((void**)&p->csr_lo, clo.data(), clo.size() * sizeof(int)); if (rc) return rc;
        rc = upload((void**)&p->csr_frac, cfr.data(), cfr.size() * sizeof(float)); if (rc) return rc;
    }
    // fused-path tables: orphan target bins (fed by no resolution) are written as zero by resolution 0
    for (int r = 0; r < d->n_res; ++r) {
        ResInfo& ri = p->res[r];
        int mn = 1 << 30, mx = -1;
        for (int l : lo[r]) { if (l < mn) mn = l; if (l > mx) mx = l; }
        if (mx >= 0) { ri.need_lo = mn; ri.need_cnt = mx + 2 - mn; } else { ri.need_lo = 0; ri.need_cnt = 0; }
        if (r == 0)
            for (int t = 0; t < d->target_bins; ++t)
                if (owners[t] == 0) { idx[0].push_back(t); lo[0].push_back(-1); fr[0].push_back(0.f); }
        ri.n_tb = (int)idx[r].size();
        int rc = upload((void**)&ri.tb_idx, idx[r].data(), idx[r].size() * sizeof(int)); if (rc) return rc;
        rc = upload((void**)&ri.tb_lo, lo[r].data(), lo[r].size() * sizeof(int)); if (rc) return rc;
        rc = upload((void**)&ri.tb_frac, fr[r].data(), fr[r].size() * sizeof(float)); if (rc) return rc;
    }
    // hop-block partial DFT path for resolutions whose combine segments read only a few FFT bins and
    // whose window is a short cosine sum: one set for the fp32 CUDA-core GEMM, one for the tensor cores
    if (p->disjoint) {
        int rc = build_sparse_set(p, d, idx, lo, false, &p->set_cc); if (rc) return rc;
        rc = build_sparse_set(p, d, idx, lo, true, &p->set_tc); if (rc) return rc;
    }
    // meters
    int rc = upload((void**)&p->hann64, d->meter_hann, (size_t)p->W * sizeof(double)); if (rc) return rc;
    std::vector<float> h32(p->W);
    for (int i = 0; i < p->W; ++i) h32[i] = (float)d->meter_hann[i];
    rc = upload((void**)&p->hann32, h32.data(), h32.size() * sizeof(float)); if (rc) return rc;
    build_biquad(d->kw_coeffs + 0, d->kw_coeffs + 3, 2, &p->kw_default[0]);
    build_biquad(d->kw_coeffs + 6, d->kw_coeffs + 9, 2, &p->kw_default[1]);
    set_weighting_k(p);
    rc = get_twiddles(p->device, ilog2(p->W), &p->tw_meter); if (rc) return rc;
    {
        const int W = p->W;
        std::vector<float2> rot((size_t)3 * W);
        const double two_pi = 6.283185307179586476925287;
        for (int ph = 1; ph <= 3; ++ph)
            for (int k = 0; k < W; ++k) {
                float2 v;
                if (k == W / 2) v = make_float2((float)cos(two_pi * ph / 8.0), 0.f);
                else {
                    const double f = (k < W / 2) ? (double)k : (double)k - W;
                    const double ang = two_pi * f * ph / (4.0 * W);
                    v = make_float2((float)cos(ang), (float)sin(ang));
                }
                rot[(size_t)(ph - 1) * W + k] = v;
            }
        rc = upload((void**)&p->tp_rot, rot.data(), rot.size() * sizeof(float2)); if (rc) return rc;
        std::vector<unsigned> roth(rot.size());
        for (size_t i = 0; i < rot.size(); ++i) {
            const __half2 h = __floats2half2_rn(rot[i].x, rot[i].y);
            memcpy(&roth[i], &h, sizeof(unsigned));
        }
        rc = upload((void**)&p->tp_rot_h, roth.data(), roth.size() * sizeof(unsigned)); if (rc) return rc;
    }
    return OMEGA4_OK;
}

extern "C" omega4_plan* omega4_plan_create(const omega4_plan_desc* desc, int device) {
    if (!desc) { fail(OMEGA4_ERR_INVALID, "desc is NULL"); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback");
        return nullptr;
    }
    if (device < 0 || device >= ndev) { fail(OMEGA4_ERR_INVALID, "bad device index"); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { fail(OMEGA4_ERR_CUDA, "cudaSetDevice failed"); return nullptr; }
    omega4_plan* p = new omega4_plan();
    p->device = device;
    if (const char* e = getenv("OMEGA4_TENSOR")) p->tensor_default = atoi(e) != 0;
    if (const char* e = getenv("OMEGA4_HOST_CHUNK_MB")) {           // tuning knob of the host-buffer pipeline
        long mb = atol(e);
        if (mb >= 16 && mb <= 16384) p->host_chunk_bytes = (size_t)mb << 20;
    }
    if (plan_build(p, desc) != OMEGA4_OK) { std::string keep = g_err; omega4_plan_destroy(p); g_err = keep; return nullptr; }
    return p;
}

static void stream_ctx_release(omega4_plan* p);

extern "C" void omega4_plan_destroy(omega4_plan* p) {
    if (!p) return;
    cudaSetDevice(p->device);
    stream_ctx_release(p);
    for (int r = 0; r < OMEGA4_MAX_RES; ++r) {
        ResInfo& ri = p->res[r];
        cudaFree(ri.window); cudaFree(ri.binw); cudaFree(ri.tb_idx); cudaFree(ri.tb_lo); cudaFree(ri.tb_frac);
        p->scratch_mag[r].release(); p->h_mag[r].release();
    }
    cudaFree(p->csr_ptr); cudaFree(p->csr_res); cudaFree(p->csr_lo); cudaFree(p->csr_frac);
    cudaFree(p->hann64); cudaFree(p->hann32); cudaFree(p->tp_rot); cudaFree(p->tp_rot_h);
    p->scratch_lufs.release(); p->scratch_tp.release(); p->scratch_q.release(); p->scratch_f32.release(); p->scratch_inv.release();
    p->scratch_comb.release(); p->scratch_bstate.release();
    p->set_cc.release(); p->set_tc.release();
    p->h_in.release(); p->h_comb.release(); p->h_meters.release(); p->h_state.release();
    p->h_f64a.release(); p->h_f64b.release(); p->h_f64c.release();
    for (auto& sl : p->slots) {
        sl.in.release(); sl.comb.release(); sl.met.release(); sl.lufs.release(); sl.tp.release(); sl.state.release();
        sl.q.release(); sl.in16.release(); sl.sc.release();
        sl.bars.release(); sl.peaks.release(); sl.bstate.release(); sl.bstate_copy.release();
        for (auto& m : sl.mag) m.release();
        if (sl.s) cudaStreamDestroy(sl.s);
    }
    for (auto& t : p->times) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
    p->sc.release();
    cudaGetLastError();
    delete p;
}

extern "C" long long omega4_plan_launches(const omega4_plan* p) { return p ? p->launches : 0; }

extern "C" int omega4_plan_set_weighting(omega4_plan* p, const omega4_weighting* w) {
    if (!p) return fail(OMEGA4_ERR_INVALID, "plan is NULL");
    if (!w) { set_weighting_k(p); return OMEGA4_OK; }
    if (w->n_sections < 0 || w->n_sections > 4) return fail(OMEGA4_ERR_INVALID, "0..4 weighting sections");
    if (w->blend && w->n_sections != 2) return fail(OMEGA4_ERR_INVALID, "the K blend needs exactly two sections");
    KwBiquad tmp[4];
    for (int i = 0; i < w->n_sections; ++i) {
        const int order = w->order[i];
        if (order != 1 && order != 2) return fail(OMEGA4_ERR_UNSUPPORTED, "weighting sections must be first or second order");
        if (w->a[i][0] == 0.0 || w->a[i][1] == 0.0 || (order == 2 && w->a[i][2] == 0.0))
            return fail(OMEGA4_ERR_UNSUPPORTED, "weighting sections need non-zero denominator coefficients");
        build_biquad(w->b[i], w->a[i], order, &tmp[i]);
    }
    for (int i = 0; i < w->n_sections; ++i) p->kw[i] = tmp[i];
    p->kw_nsec = w->n_sections; p->kw_blend = w->blend ? 1 : 0; p->kw_gate = w->rms_gate ? 1 : 0;
    p->kw_gain = w->blend ? 1.0 : w->gain;
    return OMEGA4_OK;
}

// event bracket helper
struct Bracket {
    omega4_plan* p; cudaStream_t s; bool on; KernelTime* kt = nullptr;
    Bracket(omega4_plan* p_, cudaStream_t s_, bool on_, const char* name) : p(p_), s(s_), on(on_) {
        p->launches++;
        if (!on) return;
        if (p->n_times == p->times.size()) {
            KernelTime t; memset(&t, 0, sizeof t);
            cudaEventCreate(&t.e0); cudaEventCreate(&t.e1);
            p->times.push_back(t);
        }
        kt = &p->times[p->n_times++];
        snprintf(kt->name, sizeof kt->name, "%s", name);
        cudaEventRecord(kt->e0, s);
    }
    ~Bracket() { if (on && kt) cudaEventRecord(kt->e1, s); }
};

extern "C" int omega4_plan_kernel_times(omega4_plan* p, char* names, float* ms, int max_n) {
    if (!p) return fail(OMEGA4_ERR_INVALID, "plan is NULL");
    int n = 0;
    for (size_t i = 0; i < p->n_times && n < max_n; ++i, ++n) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, p->times[i].e0, p->times[i].e1) != cudaSuccess) { cudaGetLastError(); t = -1.f; }
        if (names) { memcpy(names + 32 * n, p->times[i].name, 32); }
        if (ms) ms[n] = t;
    }
    return n;
}

// ------------------------------------------------------------------------------------------
// the hot path on device pointers
// ------------------------------------------------------------------------------------------
template <int BN>
static int launch_blockdft_gemm_t(const BlockDftGemmArgs& a, cudaStream_t s) {
    const size_t smem = blockdft_gemm_smem_bytes<BN>();
    CK(cudaFuncSetAttribute(blockdft_gemm_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long grid = (long long)((a.nb + BD_BM - 1) / BD_BM) * a.n_ch;
    if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "blockdft grid too large");
    blockdft_gemm_kernel<BN><<<(unsigned)grid, BD_THREADS, smem, s>>>(a);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

static int launch_blockdft_gemm(int bn, const BlockDftGemmArgs& a, cudaStream_t s) {
    if (a.nb <= 0 || a.n_ch <= 0) return OMEGA4_OK;
    switch (bn) {
        case 32: return launch_blockdft_gemm_t<32>(a, s);
        case 64: return launch_blockdft_gemm_t<64>(a, s);
        case 128: return launch_blockdft_gemm_t<128>(a, s);
    }
    return fail(OMEGA4_ERR_INVALID, "bad blockdft column tile");
}

static int analyze_device(omega4_plan* p, cudaStream_t s, const float* x, long long ch_stride, int n_ch,
                          int n_hops, int hist, float* combined, float* const* mags, float* meters,
                          double* lufs, double* tp, double* state, int flags, DevBuf* qbuf, SideCtx* sc) {
    const bool timing = (flags & OMEGA4_FLAG_TIME_KERNELS) != 0;
    if (timing) p->n_times = 0;
    if (((uintptr_t)x & 15) != 0 || (ch_stride % 4) != 0)
        return fail(OMEGA4_ERR_INVALID, "samples must be 16-byte aligned with ch_stride a multiple of 4");
    const bool want_meters = meters || lufs || tp;
    const bool concurrent = want_meters && (flags & OMEGA4_FLAG_CONCURRENT_METERS);
    // default: the deque-statistics kernel (one warp per channel, latency bound, few resources) runs on a
    // side stream underneath the FFT kernels that follow on the caller's stream
    const bool stats_aside = !concurrent && meters && combined && !(flags & OMEGA4_FLAG_SERIAL_STATS);
    cudaStream_t ms = s;                      // stream of the K-weighting kernel
    cudaStream_t ss = s;                      // stream of the statistics kernel
    if (concurrent || stats_aside) {
        int rc = sc->ensure(); if (rc) return rc;
        ss = sc->side;
    }
    if (concurrent) {
        ms = sc->side;
        CK(cudaEventRecord(sc->ev_fork, s));
        CK(cudaStreamWaitEvent(ms, sc->ev_fork, 0));
    }
    // ---- which resolutions the hop-block GEMM serves, and its row range (needed before the meters: the K-weighting
    // kernel can write the GEMM's per-row operand scales as a by-product)
    const bool fused = p->disjoint;
    int first[OMEGA4_MAX_RES];
    bool use_sparse[OMEGA4_MAX_RES] = {false};
    bool any_sparse = false;
    const bool tensor = p->set_tc.n > 0 && (p->tensor_default ? !(flags & OMEGA4_FLAG_NO_TENSOR) : (flags & OMEGA4_FLAG_TENSOR) != 0);
    const SparseSet& set = tensor ? p->set_tc : p->set_cc;
    for (int r = 0; r < p->n_res; ++r) {
        use_sparse[r] = combined && fused && set.of_res[r] >= 0 && !(mags && mags[r]) &&
                        !(flags & OMEGA4_FLAG_NO_BLOCKDFT);
        any_sparse = any_sparse || use_sparse[r];
        // resolution r is filled once hist + (k+1) hop >= N
        long long need = (long long)p->res[r].n - hist;
        first[r] = need <= 0 ? 0 : (int)((need + p->hop - 1) / p->hop - 1);
    }
    int sp_j0 = 1 << 30;
    for (int r = 0; r < p->n_res; ++r)
        if (use_sparse[r]) { const int j = first[r] + 1 - set.sp[set.of_res[r]].B; if (j < sp_j0) sp_j0 = j; }
    const int sp_nb = any_sparse ? n_hops - sp_j0 : 0;
    float* row_inv = nullptr;                 // [n_ch][sp_nb] operand scales of the tensor-core GEMM's hop-block rows
    int inv_from_kw = -1;                     // >= 0: the K-weighting kernel wrote the scales of hop blocks >= this index
#if TC_F16
    if (tensor && any_sparse && sp_nb > 0) {
        int rc = p->scratch_inv.ensure((size_t)n_ch * sp_nb * sizeof(float)); if (rc) return rc;
        row_inv = (float*)p->scratch_inv.p;
    }
#endif
    // ---- meters first: K-weighting on the meter stream, true peak on the caller's stream
    if (want_meters) {
        const size_t nser = (size_t)n_ch * n_hops * sizeof(double);
        if (!lufs) { int rc = p->scratch_lufs.ensure(nser); if (rc) return rc; lufs = (double*)p->scratch_lufs.p; }
        if (!tp) { int rc = p->scratch_tp.ensure(nser); if (rc) return rc; tp = (double*)p->scratch_tp.p; }
        long long need = (long long)p->W - hist;
        const int first_m = need <= 0 ? 0 : (int)((need + p->hop - 1) / p->hop - 1);
        if (use_kweight32(p)) {
            Kweight32Args k;
            memset(&k, 0, sizeof k);
            k.x = x; k.ch_stride = ch_stride; k.frame_stride = p->hop;
            k.frame_off0 = (long long)p->hop - p->W;
            k.n_ch = n_ch; k.n_frames = n_hops; k.first_frame = first_m;
            k.frames_per_warp = n_hops >= 64 ? 8 : (n_hops >= 8 ? 2 : 1);
            k.hann = p->hann32; k.lufs_out = lufs; k.rms_gate = p->kw_gate;
            if (row_inv && !concurrent && p->hop * 4 == p->W && first_m < n_hops && !getenv("OMEGA4_NO_SCALE_FOLD")) {
                k.hop_inv = row_inv; k.hop_inv_nb = sp_nb; k.hop_inv_j0 = sp_j0;       // frame f ends with hop block f
                inv_from_kw = first_m;
            }
            build_kw32(p->kw[0], &k.s[0]); build_kw32(p->kw[1], &k.s[1]);
            Bracket b(p, ms, timing, "kweight_lufs");
            int rc = launch_kweight32(k, ms);
            if (rc) return rc;
        } else {
            KweightArgs k;
            memset(&k, 0, sizeof k);
            k.x = x; k.x_is_f64 = 0; k.ch_stride = ch_stride; k.frame_stride = p->hop;
            k.frame_off0 = (long long)p->hop - p->W;
            k.n_ch = n_ch; k.n_frames = n_hops; k.first_frame = first_m;
            k.frames_per_warp = n_hops >= 64 ? 8 : (n_hops >= 8 ? 2 : 1);
            k.hann = p->hann64; k.lufs_out = lufs; k.weighted_out = nullptr;
            fill_weighting(p, &k);
            Bracket b(p, ms, timing, "kweight_lufs");
            int rc = launch_kweight(k, ms);
            if (rc) return rc;
        }
        {
            TruePeakArgs t;
            memset(&t, 0, sizeof t);
            t.x = x; t.x_is_f64 = 0; t.ch_stride = ch_stride; t.frame_stride = p->hop;
            t.frame_off0 = (long long)p->hop - p->W;
            t.n_ch = n_ch; t.n_frames = n_hops; t.first_frame = first_m;
            t.rounds = default_rounds((n_hops + 1) / 2, 2);
            t.window = p->hann32; t.twM = p->tw_meter.twM; t.rot = p->tp_rot; t.rot_h = p->tp_rot_h;
            fill_truepeak_steps(&t);
            t.tp_out = tp;
            Bracket b(p, s, timing, "true_peak");
            const bool exact_tp = (flags & OMEGA4_FLAG_EXACT_TRUE_PEAK) || getenv("OMEGA4_TP_F32");
            int rc = exact_tp ? launch_truepeak(t, s) : launch_truepeak16(t, s);
            if (rc) return rc;
        }
        if (meters) {
            if (concurrent || stats_aside) {
                CK(cudaEventRecord(sc->ev_tp, s));
                CK(cudaStreamWaitEvent(ss, sc->ev_tp, 0));
            }
            StatsArgs st;
            memset(&st, 0, sizeof st);
            st.lufs = lufs; st.tp = tp; st.n_ch = n_ch; st.n_frames = n_hops; st.first_frame = first_m;
            st.gate = p->gate; st.out = meters;
            st.fresh = (state == nullptr) || (flags & OMEGA4_FLAG_FRESH_METERS) ? 1 : 0;
            if (!state) {
                int rc = p->h_state.ensure((size_t)n_ch * ST_STATE * sizeof(double));
                if (rc) return rc;
                state = (double*)p->h_state.p;
            }
            st.state = state;
            Bracket b(p, ss, timing, "meter_stats");
            int rc = launch_stats(st, ss);
            if (rc) return rc;
        }
        if (concurrent || stats_aside) CK(cudaEventRecord(sc->ev_join, ss));
    }
    // ---- multi-resolution FFTs (+ fused combine) on the caller's stream
    float* mag_ptr[OMEGA4_MAX_RES];
    for (int r = 0; r < p->n_res; ++r) {
        ResInfo& ri = p->res[r];
        mag_ptr[r] = mags ? mags[r] : nullptr;
        if (combined && !fused && !mag_ptr[r]) {
            int rc = p->scratch_mag[r].ensure((size_t)n_ch * n_hops * ri.bins * sizeof(float));
            if (rc) return rc;
            mag_ptr[r] = (float*)p->scratch_mag[r].p;
        }
        if (!combined && !mag_ptr[r]) continue;
        if (use_sparse[r]) continue;                      // served by the hop-block partial DFT below
        MultiresArgs a;
        memset(&a, 0, sizeof a);
        a.x = x; a.ch_stride = ch_stride; a.frame_stride = p->hop; a.frame_off0 = (long long)p->hop - ri.n;
        a.n_ch = n_ch; a.n_frames = n_hops; a.first_frame = first[r];
        a.rounds = default_rounds(n_hops, (1 << ri.log2m) >= 4096 ? 1 : 4096 >> ri.log2m);
        a.window = ri.window; a.binw = ri.binw; a.twM = ri.tw.twM; a.twN = ri.tw.twN;
        a.mag_out = mag_ptr[r]; a.cplx_out = nullptr;
        a.comb_out = (combined && fused) ? combined : nullptr;
        a.T = p->T; a.n_tb = ri.n_tb; a.tb_idx = ri.tb_idx; a.tb_lo = ri.tb_lo; a.tb_frac = ri.tb_frac;
        a.wnum = ri.weight; a.wden = ri.weight;
        a.need_lo = ri.need_lo; a.need_cnt = (combined && fused) ? ri.need_cnt : 0;
        char name[32];
        snprintf(name, sizeof name, "multires_fft_%d", ri.n);
        Bracket b(p, s, timing, name);
        int rc = launch_multires(ri.log2m, a, s);
        if (rc) return rc;
    }
    if (any_sparse) {
        // one GEMM over the hop blocks serves every sparse resolution; then one assembly per resolution
        const int j0 = sp_j0, nb = sp_nb;
        const float* Q = nullptr;
        const bool fusedx = tensor && set.fusable;        // frames assembled in the GEMM epilogue, no Q
        if (nb > 0) {
            const size_t qbytes = fusedx ? (size_t)n_ch * set.nkx * n_hops * sizeof(float2)
                                         : (size_t)n_ch * nb * set.qs * sizeof(float);
            int rc = qbuf->ensure(qbytes);
            if (rc) return rc;
            Q = (float*)qbuf->p;
            if (tensor) {
                BlockDftTcArgs g;
                memset(&g, 0, sizeof g);
                g.x = x; g.ch_stride = ch_stride; g.hop = p->hop; g.n_ch = n_ch; g.j0 = j0; g.nb = nb;
                g.n_halves = set.n_halves; g.Eimg = set.Eimg; g.Q = (float*)qbuf->p; g.qs = set.qs;
#if TC_F16
                {   // per hop-block row operand scale (half's exponent range is spent below each row's own maximum)
                    HopScaleArgs h;
                    h.x = x; h.ch_stride = ch_stride; h.hop = p->hop; h.n_ch = n_ch; h.j0 = j0; h.nb = nb;
                    // hop blocks from inv_from_kw on have their scale from the K-weighting kernel of this call
                    h.ncols = inv_from_kw >= 0 ? inv_from_kw - j0 : nb;
                    h.inv = row_inv;
                    g.row_inv = h.inv; g.e_inv = set.e_inv;
                    const long long rows = (long long)n_ch * h.ncols;
                    if (rows > 0) {
                        Bracket b(p, s, timing, "blockdft_row_scale");
                        hopblock_scale_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(h);
                        CK(cudaGetLastError());
                    }
                }
#endif
                if (fusedx) {
                    g.X = (float2*)qbuf->p; g.n_frames = n_hops; g.nkx = set.nkx;
                    memcpy(g.gB, set.gB, sizeof g.gB); memcpy(g.gX, set.gX, sizeof g.gX); memcpy(g.gN, set.gN, sizeof g.gN);
                    memcpy(g.gS, set.gS, sizeof g.gS);
                    CK(cudaMemsetAsync(qbuf->p, 0, qbytes, s));      // frames that straddle row tiles are completed with atomics
                }
                const size_t smem = blockdft_tc_smem_bytes();
                CK(cudaFuncSetAttribute(blockdft_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                const long long n_tiles = (long long)((nb + TC_BM - 1) / TC_BM) * n_ch * set.n_halves;
                if (n_tiles > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "blockdft grid too large");
                g.n_tiles = (int)n_tiles;
                // persistent: one CTA per SM walks over the tiles (b, b + grid, ...; the column tiles of a row tile run
                // side by side on neighbouring SMs, so the samples are read from HBM once)
                static int n_sm = 0;
                if (!n_sm) { int dev = 0; CK(cudaGetDevice(&dev)); CK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev)); }
                const bool persistent = !getenv("OMEGA4_TC_ONE_TILE_PER_CTA");
                const long long grid = persistent ? std::min<long long>(n_tiles, n_sm) : n_tiles;
                Bracket b(p, s, timing, "blockdft_tc_gemm");
                blockdft_tc_kernel<<<(unsigned)grid, TC_CTA_THREADS, smem, s>>>(g);
                CK(cudaGetLastError());
#ifdef TC_TIMELINE
                {   // developer builds: phase durations (cycles) of the second tile of every 4th CTA, median over the sampled CTAs
                    static long long h[64][16];
                    CK(cudaStreamSynchronize(s));
                    CK(cudaMemcpyFromSymbol(h, tc_tl, sizeof h));
                    const int n = (int)std::min<long long>(64, (grid + 3) / 4);
                    const char* nm[12] = {"wait_empty+operands", "mma_issue_loop", "commit->full_seen", "tmem_drain", "epilogue_rest", "tile_period",
                                          "cg2 wait::ld", "cg2 acc+sts", "cg2 ld issue", "cg2 bar1", "cg2 sums", "cg2 bar2"};
                    const int from[12] = {0, 1, 2, 3, 4, 0, 8, 9, 10, 11, 12, 13}, to[12] = {1, 2, 3, 4, 5, 6, 9, 10, 11, 12, 13, 14};
                    for (int k = 0; k < 12; ++k) {
                        std::vector<long long> d;
                        for (int i = 0; i < n; ++i) d.push_back(h[i][to[k]] - h[i][from[k]]);
                        std::sort(d.begin(), d.end());
                        fprintf(stderr, "tc_timeline %-20s median %lld  p10 %lld  p90 %lld\n", nm[k], d[n / 2], d[n / 10], d[n * 9 / 10]);
                    }
                }
#endif
            } else {
                BlockDftGemmArgs g;
                memset(&g, 0, sizeof g);
                g.x = x; g.ch_stride = ch_stride; g.hop = p->hop; g.n_ch = n_ch; g.j0 = j0; g.nb = nb;
                g.E = set.E; g.Q = (float*)qbuf->p;
                Bracket b(p, s, timing, "blockdft_gemm");
                rc = launch_blockdft_gemm(set.qs, g, s);
                if (rc) return rc;
            }
        }
        for (int r = 0; r < p->n_res; ++r) {
            if (!use_sparse[r]) continue;
            const ResInfo& ri = p->res[r];
            const SparseRes& sp = set.sp[set.of_res[r]];
            if (sp.td && fusedx) {
                BlockDftFinishArgs a;
                memset(&a, 0, sizeof a);
                a.X = (const float2*)Q; a.nkx = set.nkx; a.xoff = sp.xoff; a.nk = sp.nk; a.kw = sp.kw;
                a.n_ch = n_ch; a.n_frames = n_hops; a.first_frame = first[r];
                a.comb_out = combined; a.Tbins = p->T; a.n_tb = ri.n_tb; a.tb_idx = ri.tb_idx; a.tb_pos = sp.tb_pos;
                a.tb_frac = ri.tb_frac; a.wnum = ri.weight; a.wden = ri.weight;
                const size_t smem = blockdft_finish_smem_bytes(sp.nk);
                CK(cudaFuncSetAttribute(blockdft_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                const long long grid = (long long)((n_hops + BD_FIN_FRAMES - 1) / BD_FIN_FRAMES) * n_ch;
                if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "blockdft finish grid too large");
                char name[32];
                snprintf(name, sizeof name, "blockdft_asm_%d", ri.n);
                Bracket b(p, s, timing, name);
                blockdft_finish_kernel<<<(unsigned)grid, 256, smem, s>>>(a);
                CK(cudaGetLastError());
                continue;
            }
            if (sp.td) {
                BlockDftSumArgs a;
                memset(&a, 0, sizeof a);
                a.Q = Q; a.qs = set.qs; a.col0 = sp.col0; a.nb = nb > 0 ? nb : 0; a.j0 = j0;
                a.nk = sp.nk; a.B = sp.B; a.kw = sp.kw;
                a.n_ch = n_ch; a.n_frames = n_hops; a.first_frame = first[r];
                a.comb_out = combined; a.Tbins = p->T; a.n_tb = ri.n_tb; a.tb_idx = ri.tb_idx; a.tb_pos = sp.tb_pos;
                a.tb_frac = ri.tb_frac; a.wnum = ri.weight; a.wden = ri.weight;
                a.fa = blockdft_sum_frames(sp.nk, sp.B);
                const size_t smem = blockdft_sum_smem_bytes(sp.nk, sp.B, a.fa);
                CK(cudaFuncSetAttribute(blockdft_sum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                const long long grid = (long long)((n_hops + a.fa - 1) / a.fa) * n_ch;
                if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "blockdft assemble grid too large");
                char name[32];
                snprintf(name, sizeof name, "blockdft_asm_%d", ri.n);
                Bracket b(p, s, timing, name);
                blockdft_sum_kernel<<<(unsigned)grid, 256, smem, s>>>(a);
                CK(cudaGetLastError());
                continue;
            }
            BlockDftAsmArgs a;
            memset(&a, 0, sizeof a);
            a.Q = Q; a.qs = set.qs; a.col0 = sp.col0; a.nb = nb > 0 ? nb : 0; a.j0 = j0;
            a.nk = sp.nk; a.nt = sp.nt; a.B = sp.B; a.T = sp.T; a.kw = sp.kw;
            a.n_ch = n_ch; a.n_frames = n_hops; a.first_frame = first[r];
            a.comb_out = combined; a.Tbins = p->T; a.n_tb = ri.n_tb; a.tb_idx = ri.tb_idx; a.tb_pos = sp.tb_pos;
            a.tb_frac = ri.tb_frac; a.wnum = ri.weight; a.wden = ri.weight;
            a.fa = blockdft_assemble_frames(sp.nk, sp.nt, sp.B);
            const size_t smem = blockdft_assemble_smem_bytes(sp.nk, sp.nt, sp.B, a.fa);
            auto kern = sp.nt == 5 ? blockdft_assemble_kernel<5> : (sp.nt == 3 ? blockdft_assemble_kernel<3> : blockdft_assemble_kernel<1>);
            CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const long long grid = (long long)((n_hops + a.fa - 1) / a.fa) * n_ch;
            if (grid > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "blockdft assemble grid too large");
            char name[32];
            snprintf(name, sizeof name, "blockdft_asm_%d", ri.n);
            Bracket b(p, s, timing, name);
            kern<<<(unsigned)grid, 256, smem, s>>>(a);
            CK(cudaGetLastError());
        }
    }
    if (combined && !fused) {
        CombineArgs c;
        memset(&c, 0, sizeof c);
        for (int r = 0; r < p->n_res; ++r) {
            c.mag[r] = mag_ptr[r]; c.bins[r] = p->res[r].bins; c.first_frame[r] = first[r]; c.weight[r] = p->res[r].weight;
        }
        c.n_hops = n_hops; c.n_rows = n_ch * n_hops; c.T = p->T;
        c.csr_ptr = p->csr_ptr; c.csr_res = p->csr_res; c.csr_lo = p->csr_lo; c.csr_frac = p->csr_frac;
        c.out = combined;
        const long long total = (long long)c.n_rows * c.T;
        Bracket b(p, s, timing, "combine");
        combine_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(c);
        CK(cudaGetLastError());
    }
    if (concurrent || stats_aside) CK(cudaStreamWaitEvent(s, sc->ev_join, 0));
    return OMEGA4_OK;
}

// s16 != nullptr: the input is interleaved little-endian int16 (capture.py:571-574), `il` channels per
// stream, stream g starting at s16 + g*ch_stride (int16 units, pointing at the first NEW frame;
// hist_samples frames precede it); n_ch = streams * il planar channels come out of the conversion.
static int analyze_any(omega4_plan* p, void* stream, int mem, const float* samples, const int16_t* s16, int il,
                       long long ch_stride, int n_ch, int n_hops, int hist_samples, float* combined,
                       float* const* magnitudes, float* meters, double* lufs_inst, double* tp_db,
                       double* meter_state, int flags, const BarsReq* br = nullptr) {
    if (!p) return fail(OMEGA4_ERR_INVALID, "plan is NULL");
    if (br && !br->b) br = nullptr;
    if (br) {
        if (!br->band_values) return fail(OMEGA4_ERR_INVALID, "band_values is NULL");
        if (br->b->device != p->device || br->b->T != p->T)
            return fail(OMEGA4_ERR_INVALID, "the bars object must live on the plan's device and take spectra of target_bins values");
    }
    if ((!samples && !s16) || n_ch < 0 || n_hops < 0 || hist_samples < 0) return fail(OMEGA4_ERR_INVALID, "bad samples / sizes");
    if (s16 && (il < 1 || il > 64 || n_ch % il != 0)) return fail(OMEGA4_ERR_INVALID, "bad interleave");
    if (n_ch == 0 || n_hops == 0) return OMEGA4_OK;
    CK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (mem == OMEGA4_MEM_DEVICE) {
        if (s16) {
            const long long hist_al = ((long long)hist_samples + 3) / 4 * 4;
            const long long len = (long long)hist_samples + (long long)n_hops * p->hop;
            const long long dstride = (hist_al + (long long)n_hops * p->hop + 3) / 4 * 4;
            int rc = p->scratch_f32.ensure((size_t)n_ch * dstride * sizeof(float)); if (rc) return rc;
            float* d_in = (float*)p->scratch_f32.p;
            p->launches++;
            rc = launch_s16_convert(s16 - (long long)hist_samples * il, ch_stride, il, n_ch / il, len,
                                    d_in + (hist_al - hist_samples), dstride, s);
            if (rc) return rc;
            samples = d_in + hist_al; ch_stride = dstride;
        }
        float* d_comb = combined;
        if (br && !d_comb) {
            int rc = p->scratch_comb.ensure((size_t)n_ch * n_hops * p->T * sizeof(float)); if (rc) return rc;
            d_comb = (float*)p->scratch_comb.p;
        }
        int rc = analyze_device(p, s, samples, ch_stride, n_ch, n_hops, hist_samples, d_comb, magnitudes, meters,
                                lufs_inst, tp_db, meter_state, flags, &p->scratch_q, &p->sc);
        if (rc || !br) return rc;
        p->launches++;
        return bars_launch(br->b, s, d_comb, n_ch, n_hops, br->state, br->fresh, br->band_values, br->peak_values, &p->scratch_bstate);
    }
    if (mem != OMEGA4_MEM_HOST) return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");

    // ---- host buffers: channel chunks pipelined over private streams (H2D | kernels | D2H overlap)
    CK(cudaStreamSynchronize(s));                                  // order after the caller's stream
    const long long hist = hist_samples;
    const long long hist_al = (hist + 3) / 4 * 4;                 // keep device rows 16-byte aligned
    const long long new_len = (long long)n_hops * p->hop;
    const long long dstride = (hist_al + new_len + 3) / 4 * 4;
    size_t per_ch = (size_t)dstride * sizeof(float) + (size_t)n_hops * 2 * sizeof(double) + ST_STATE * sizeof(double);
    if (combined || br) per_ch += (size_t)n_hops * p->T * sizeof(float);
    if (br) per_ch += (size_t)n_hops * br->b->n_valid * sizeof(float) * (br->peak_values ? 2 : 1);
    {
        const bool tensor_sel = p->set_tc.n > 0 && (p->tensor_default ? !(flags & OMEGA4_FLAG_NO_TENSOR) : (flags & OMEGA4_FLAG_TENSOR) != 0);
        const SparseSet& sset = tensor_sel ? p->set_tc : p->set_cc;
        if ((combined || br) && sset.n > 0 && !(flags & OMEGA4_FLAG_NO_BLOCKDFT))
            per_ch += (tensor_sel && sset.fusable) ? (size_t)(n_hops + 64) * sset.nkx * sizeof(float2)
                                                   : (size_t)(n_hops + 64) * sset.qs * sizeof(float);
    }
    if (meters) per_ch += (size_t)n_hops * 5 * sizeof(float);
    bool want_mag[OMEGA4_MAX_RES] = {false};
    for (int r = 0; r < p->n_res; ++r) {
        want_mag[r] = (magnitudes && magnitudes[r]) || ((combined || br) && !p->disjoint);
        if (want_mag[r]) per_ch += (size_t)n_hops * p->res[r].bins * sizeof(float);
    }
    if (s16) per_ch += (size_t)(hist + new_len) * sizeof(int16_t);
    int chunk = (int)(p->host_chunk_bytes / per_ch);
    if (chunk < 1) chunk = 1;
    if (chunk > n_ch) chunk = n_ch;
    if (s16) { chunk = chunk / il * il; if (chunk < il) chunk = il; }     // whole streams per chunk
    const bool want_series = meters || lufs_inst || tp_db;
    int idx = 0;
    for (int c0 = 0; c0 < n_ch; c0 += chunk, ++idx) {
        const int nc = (n_ch - c0 < chunk) ? n_ch - c0 : chunk;
        omega4_plan::Slot& sl = p->slots[idx % omega4_plan::N_SLOTS];
        if (!sl.s) CK(cudaStreamCreateWithFlags(&sl.s, cudaStreamNonBlocking));
        const size_t rows = (size_t)nc * n_hops;
        int rc = sl.in.ensure((size_t)nc * dstride * sizeof(float)); if (rc) return rc;
        float* d_in = (float*)sl.in.p;
        if (s16) {
            const int ns = nc / il;                                   // streams in this chunk
            const size_t row16 = (size_t)(hist + new_len) * il;       // int16 per stream
            rc = sl.in16.ensure((size_t)ns * row16 * sizeof(int16_t)); if (rc) return rc;
            CK(cudaMemcpy2DAsync(sl.in16.p, row16 * sizeof(int16_t),
                                 s16 + (long long)(c0 / il) * ch_stride - hist * il, ch_stride * sizeof(int16_t),
                                 row16 * sizeof(int16_t), ns, cudaMemcpyHostToDevice, sl.s));
            p->launches++;
            rc = launch_s16_convert((const int16_t*)sl.in16.p, (long long)row16, il, ns, hist + new_len,
                                    d_in + (hist_al - hist), dstride, sl.s);
            if (rc) return rc;
        } else {
            CK(cudaMemcpy2DAsync(d_in + (hist_al - hist), dstride * sizeof(float),
                                 samples + (long long)c0 * ch_stride - hist, ch_stride * sizeof(float),
                                 (size_t)(hist + new_len) * sizeof(float), nc, cudaMemcpyHostToDevice, sl.s));
        }
        float* d_comb = nullptr; float* d_met = nullptr; double* d_state = nullptr;
        double* d_lufs = nullptr; double* d_tp = nullptr;
        float* d_mag[OMEGA4_MAX_RES] = {nullptr};
        if (combined || br) { rc = sl.comb.ensure(rows * p->T * sizeof(float)); if (rc) return rc; d_comb = (float*)sl.comb.p; }
        float* d_bars = nullptr; float* d_peaks = nullptr; float* d_bstate = nullptr;
        const size_t bst_row = br ? (size_t)(1 + br->b->n_valid) : 0;
        if (br) {
            rc = sl.bars.ensure(rows * br->b->n_valid * sizeof(float)); if (rc) return rc; d_bars = (float*)sl.bars.p;
            if (br->peak_values) { rc = sl.peaks.ensure(rows * br->b->n_valid * sizeof(float)); if (rc) return rc; d_peaks = (float*)sl.peaks.p; }
            if (br->state) {
                rc = sl.bstate.ensure((size_t)nc * bst_row * sizeof(float)); if (rc) return rc; d_bstate = (float*)sl.bstate.p;
                if (!br->fresh)
                    CK(cudaMemcpyAsync(d_bstate, br->state + (size_t)c0 * bst_row, (size_t)nc * bst_row * sizeof(float), cudaMemcpyHostToDevice, sl.s));
            }
        }
        if (meters) { rc = sl.met.ensure(rows * 5 * sizeof(float)); if (rc) return rc; d_met = (float*)sl.met.p; }
        if (want_series) {
            rc = sl.lufs.ensure(rows * sizeof(double)); if (rc) return rc; d_lufs = (double*)sl.lufs.p;
            rc = sl.tp.ensure(rows * sizeof(double)); if (rc) return rc; d_tp = (double*)sl.tp.p;
        }
        if (meters) {
            rc = sl.state.ensure((size_t)nc * ST_STATE * sizeof(double)); if (rc) return rc;
            d_state = (double*)sl.state.p;
            if (meter_state && !(flags & OMEGA4_FLAG_FRESH_METERS))
                CK(cudaMemcpyAsync(d_state, meter_state + (size_t)c0 * ST_STATE, (size_t)nc * ST_STATE * sizeof(double),
                                   cudaMemcpyHostToDevice, sl.s));
        }
        bool any_mag = false;
        for (int r = 0; r < p->n_res; ++r)
            if (want_mag[r]) {
                rc = sl.mag[r].ensure(rows * p->res[r].bins * sizeof(float)); if (rc) return rc;
                d_mag[r] = (float*)sl.mag[r].p; any_mag = true;
            }
        const int fl = (flags & ~OMEGA4_FLAG_CONCURRENT_METERS) | ((meter_state == nullptr) ? OMEGA4_FLAG_FRESH_METERS : 0);
        rc = analyze_device(p, sl.s, d_in + hist_al, dstride, nc, n_hops, (int)hist, d_comb, any_mag ? d_mag : nullptr,
                            d_met, d_lufs, d_tp, d_state, fl, &sl.q, &sl.sc);
        if (rc) return rc;
        const size_t r0 = (size_t)c0 * n_hops;
        if (br) {
            p->launches++;
            rc = bars_launch(br->b, sl.s, d_comb, nc, n_hops, d_bstate, br->fresh, d_bars, d_peaks, &sl.bstate_copy);
            if (rc) return rc;
            const size_t nv = (size_t)br->b->n_valid;
            CK(cudaMemcpyAsync(br->band_values + r0 * nv, d_bars, rows * nv * sizeof(float), cudaMemcpyDeviceToHost, sl.s));
            if (br->peak_values) CK(cudaMemcpyAsync(br->peak_values + r0 * nv, d_peaks, rows * nv * sizeof(float), cudaMemcpyDeviceToHost, sl.s));
            if (br->state) CK(cudaMemcpyAsync(br->state + (size_t)c0 * bst_row, d_bstate, (size_t)nc * bst_row * sizeof(float), cudaMemcpyDeviceToHost, sl.s));
        }
        if (combined) CK(cudaMemcpyAsync(combined + r0 * p->T, d_comb, rows * p->T * sizeof(float), cudaMemcpyDeviceToHost, sl.s));
        if (meters) CK(cudaMemcpyAsync(meters + r0 * 5, d_met, rows * 5 * sizeof(float), cudaMemcpyDeviceToHost, sl.s));
        if (lufs_inst) CK(cudaMemcpyAsync(lufs_inst + r0, d_lufs, rows * sizeof(double), cudaMemcpyDeviceToHost, sl.s));
        if (tp_db) CK(cudaMemcpyAsync(tp_db + r0, d_tp, rows * sizeof(double), cudaMemcpyDeviceToHost, sl.s));
        if (meters && meter_state)
            CK(cudaMemcpyAsync(meter_state + (size_t)c0 * ST_STATE, d_state, (size_t)nc * ST_STATE * sizeof(double),
                               cudaMemcpyDeviceToHost, sl.s));
        if (magnitudes)
            for (int r = 0; r < p->n_res; ++r)
                if (magnitudes[r])
                    CK(cudaMemcpyAsync(magnitudes[r] + r0 * p->res[r].bins, d_mag[r], rows * p->res[r].bins * sizeof(float),
                                       cudaMemcpyDeviceToHost, sl.s));
    }
    for (auto& sl : p->slots)
        if (sl.s) CK(cudaStreamSynchronize(sl.s));
    return OMEGA4_OK;
}

extern "C" int omega4_analyze(omega4_plan* p, void* stream, int mem, const float* samples, long long ch_stride,
                              int n_ch, int n_hops, int hist_samples, float* combined, float* const* magnitudes,
                              float* meters, double* lufs_inst, double* tp_db, double* meter_state, int flags) {
    if (!samples) return fail(OMEGA4_ERR_INVALID, "bad samples / sizes");
    return analyze_any(p, stream, mem, samples, nullptr, 1, ch_stride, n_ch, n_hops, hist_samples, combined, magnitudes,
                       meters, lufs_inst, tp_db, meter_state, flags);
}

extern "C" int omega4_analyze_s16(omega4_plan* p, void* stream, int mem, const int16_t* frames, long long stream_stride,
                                  int n_streams, int n_interleaved, int n_hops, int hist_frames, float* combined,
                                  float* const* magnitudes, float* meters, double* lufs_inst, double* tp_db,
                                  double* meter_state, int flags) {
    if (!frames || n_streams < 0 || n_interleaved < 1) return fail(OMEGA4_ERR_INVALID, "bad frames / sizes");
    if (mem == OMEGA4_MEM_DEVICE && ((uintptr_t)frames & 1)) return fail(OMEGA4_ERR_INVALID, "frames must be 2-byte aligned");
    return analyze_any(p, stream, mem, nullptr, frames, n_interleaved, stream_stride, n_streams * n_interleaved, n_hops,
                       hist_frames, combined, magnitudes, meters, lufs_inst, tp_db, meter_state, flags);
}

extern "C" int omega4_analyze_io(omega4_plan* p, void* stream, int mem, const omega4_io* io) {
    if (!io) return fail(OMEGA4_ERR_INVALID, "io is NULL");
    if ((io->samples != nullptr) == (io->frames_s16 != nullptr))
        return fail(OMEGA4_ERR_INVALID, "exactly one of samples / frames_s16 must be given");
    BarsReq br;
    br.b = io->bars; br.band_values = io->band_values; br.peak_values = io->peak_values; br.state = io->bars_state;
    br.fresh = (!io->bars_state || (io->flags & OMEGA4_FLAG_FRESH_BARS)) ? 1 : 0;
    if (io->frames_s16) {
        if (io->n_interleaved < 1 || io->n_ch % io->n_interleaved != 0) return fail(OMEGA4_ERR_INVALID, "bad interleave");
        if (mem == OMEGA4_MEM_DEVICE && ((uintptr_t)io->frames_s16 & 1)) return fail(OMEGA4_ERR_INVALID, "frames must be 2-byte aligned");
        return analyze_any(p, stream, mem, nullptr, io->frames_s16, io->n_interleaved, io->stride, io->n_ch, io->n_hops, io->hist,
                           io->combined, io->magnitudes, io->meters, io->lufs_inst, io->tp_db, io->meter_state, io->flags, &br);
    }
    return analyze_any(p, stream, mem, io->samples, nullptr, 1, io->stride, io->n_ch, io->n_hops, io->hist, io->combined,
                       io->magnitudes, io->meters, io->lufs_inst, io->tp_db, io->meter_state, io->flags, &br);
}

// ------------------------------------------------------------------------------------------
// streaming entry points: one round trip per application frame
// ------------------------------------------------------------------------------------------
struct StreamCtx {
    cudaStream_t s = nullptr;
    float* h_in = nullptr; float* h_out = nullptr;       // pinned staging
    size_t h_in_cap = 0, h_out_cap = 0;
    DevBuf d_in, d_out;
    double* h64 = nullptr; size_t h64_cap = 0;            // pinned staging of the meter update
    DevBuf d64;
    std::map<unsigned, cudaGraphExec_t> graphs;           // omega4_stream_hop: one captured graph per set of ready resolutions
    std::set<unsigned> seen;
    void drop_graphs() { for (auto& kv : graphs) cudaGraphExecDestroy(kv.second); graphs.clear(); seen.clear(); }
    int ensure(size_t in_bytes, size_t out_bytes) {
        if (!s) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        if (in_bytes > h_in_cap) { if (h_in) cudaFreeHost(h_in); h_in = nullptr; h_in_cap = 0; CK(cudaMallocHost(&h_in, in_bytes)); h_in_cap = in_bytes; }
        if (out_bytes > h_out_cap) { if (h_out) cudaFreeHost(h_out); h_out = nullptr; h_out_cap = 0; CK(cudaMallocHost(&h_out, out_bytes)); h_out_cap = out_bytes; }
        int rc = d_in.ensure(in_bytes); if (rc) return rc;
        return d_out.ensure(out_bytes);
    }
    int ensure64(size_t bytes) {
        if (!s) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        if (bytes > h64_cap) { if (h64) cudaFreeHost(h64); h64 = nullptr; h64_cap = 0; CK(cudaMallocHost(&h64, bytes)); h64_cap = bytes; }
        return d64.ensure(bytes);
    }
    void release() {
        drop_graphs();
        if (h_in) cudaFreeHost(h_in); if (h_out) cudaFreeHost(h_out); if (h64) cudaFreeHost(h64);
        d_in.release(); d_out.release(); d64.release();
        if (s) cudaStreamDestroy(s);
        h_in = h_out = nullptr; h64 = nullptr; s = nullptr; h_in_cap = h_out_cap = h64_cap = 0;
    }
};
static std::mutex g_sc_mu;
static std::map<omega4_plan*, StreamCtx> g_stream_ctx;
static StreamCtx* stream_ctx(omega4_plan* p) { std::lock_guard<std::mutex> lk(g_sc_mu); return &g_stream_ctx[p]; }
static void stream_ctx_release(omega4_plan* p) {
    std::lock_guard<std::mutex> lk(g_sc_mu);
    auto it = g_stream_ctx.find(p);
    if (it != g_stream_ctx.end()) { it->second.release(); g_stream_ctx.erase(it); }
}

// enqueue one hop's work on the context's stream: H2D of the packed frames, one FFT launch per ready resolution,
// the combine over exactly those, D2H of the packed results
static int stream_hop_enqueue(omega4_plan* p, StreamCtx* c, unsigned ready, bool want_comb, const size_t* in_off,
                              const size_t* out_off, size_t in_tot, size_t out_tot, size_t comb_off) {
    CK(cudaMemcpyAsync(c->d_in.p, c->h_in, in_tot * sizeof(float), cudaMemcpyHostToDevice, c->s));
    CombineArgs cb;
    memset(&cb, 0, sizeof cb);
    for (int r = 0; r < p->n_res; ++r) {
        cb.bins[r] = p->res[r].bins; cb.first_frame[r] = 0; cb.weight[r] = p->res[r].weight;
        if (!(ready >> r & 1)) continue;
        const ResInfo& ri = p->res[r];
        MultiresArgs a;
        memset(&a, 0, sizeof a);
        a.x = (const float*)c->d_in.p + in_off[r]; a.ch_stride = 0; a.frame_stride = ri.n; a.frame_off0 = 0;
        a.n_ch = 1; a.n_frames = 1; a.first_frame = 0; a.rounds = 1;
        a.window = ri.window; a.binw = ri.binw; a.twM = ri.tw.twM; a.twN = ri.tw.twN;
        a.mag_out = (float*)c->d_out.p + out_off[r];
        int rc = launch_multires(ri.log2m, a, c->s);
        if (rc) return rc;
        cb.mag[r] = a.mag_out;
    }
    if (want_comb) {
        cb.n_hops = 0; cb.n_rows = 1; cb.T = p->T;
        cb.csr_ptr = p->csr_ptr; cb.csr_res = p->csr_res; cb.csr_lo = p->csr_lo; cb.csr_frac = p->csr_frac;
        cb.out = (float*)c->d_out.p + comb_off;
        combine_kernel<<<(unsigned)((p->T + 255) / 256), 256, 0, c->s>>>(cb);
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(c->h_out, c->d_out.p, out_tot * sizeof(float), cudaMemcpyDeviceToHost, c->s));
    return OMEGA4_OK;
}

extern "C" int omega4_stream_hop(omega4_plan* p, const float* const* frames, float* const* magnitudes, float* combined) {
    if (!p || !frames || !magnitudes) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    CK(cudaSetDevice(p->device));
    size_t in_off[OMEGA4_MAX_RES], out_off[OMEGA4_MAX_RES], in_tot = 0, out_tot = 0;
    unsigned ready = 0;
    int n_ready = 0;
    for (int r = 0; r < p->n_res; ++r) {
        in_off[r] = in_tot; out_off[r] = out_tot;
        if (frames[r]) {
            if (!magnitudes[r]) return fail(OMEGA4_ERR_INVALID, "a ready resolution needs a magnitude buffer");
            in_tot += (size_t)p->res[r].n; out_tot += ((size_t)p->res[r].bins + 3) / 4 * 4; ++n_ready; ready |= 1u << r;
        }
    }
    const size_t comb_off = out_tot;
    if (combined) out_tot += (size_t)p->T;
    if (n_ready == 0) {
        if (combined) memset(combined, 0, (size_t)p->T * sizeof(float));
        return OMEGA4_OK;
    }
    StreamCtx* c = stream_ctx(p);
    const bool grew = in_tot * sizeof(float) > c->h_in_cap || out_tot * sizeof(float) > c->h_out_cap;
    int rc = c->ensure(in_tot * sizeof(float), out_tot * sizeof(float)); if (rc) return rc;
    if (grew) c->drop_graphs();                                   // the staging buffers moved
    for (int r = 0; r < p->n_res; ++r)
        if (frames[r]) memcpy(c->h_in + in_off[r], frames[r], (size_t)p->res[r].n * sizeof(float));
    // The same set of ready resolutions recurs on every hop once the rings have filled: its copies and launches are
    // captured into a CUDA graph on the second occurrence (the first one runs eagerly and sets the kernels' attributes)
    // and replayed with one launch afterwards.  OMEGA4_STREAM_GRAPH=0 keeps the eager path.
    const unsigned key = ready | (combined ? 1u << 31 : 0u);
    static const bool use_graph = !(getenv("OMEGA4_STREAM_GRAPH") && atoi(getenv("OMEGA4_STREAM_GRAPH")) == 0);
    cudaGraphExec_t exec = nullptr;
    if (use_graph) {
        auto it = c->graphs.find(key);
        if (it != c->graphs.end()) exec = it->second;
    }
    p->launches += n_ready + (combined ? 1 : 0);
    if (exec) {
        CK(cudaGraphLaunch(exec, c->s));
    } else if (use_graph && c->seen.count(key)) {
        cudaGraph_t g = nullptr;
        CK(cudaStreamBeginCapture(c->s, cudaStreamCaptureModeThreadLocal));
        rc = stream_hop_enqueue(p, c, ready, combined != nullptr, in_off, out_off, in_tot, out_tot, comb_off);
        cudaError_t e = cudaStreamEndCapture(c->s, &g);
        if (rc) { if (g) cudaGraphDestroy(g); return rc; }
        if (e != cudaSuccess) return fail(OMEGA4_ERR_CUDA, std::string("stream capture failed: ") + cudaGetErrorString(e));
        e = cudaGraphInstantiate(&exec, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) return fail(OMEGA4_ERR_CUDA, std::string("cudaGraphInstantiate failed: ") + cudaGetErrorString(e));
        c->graphs[key] = exec;
        CK(cudaGraphLaunch(exec, c->s));
    } else {
        c->seen.insert(key);
        rc = stream_hop_enqueue(p, c, ready, combined != nullptr, in_off, out_off, in_tot, out_tot, comb_off);
        if (rc) return rc;
    }
    CK(cudaStreamSynchronize(c->s));
    for (int r = 0; r < p->n_res; ++r)
        if (frames[r]) memcpy(magnitudes[r], c->h_out + out_off[r], (size_t)p->res[r].bins * sizeof(float));
    if (combined) memcpy(combined, c->h_out + comb_off, (size_t)p->T * sizeof(float));
    return OMEGA4_OK;
}

extern "C" int omega4_meter_update(omega4_plan* p, const double* frame, double* state, int fresh, float* meters,
                                   double* lufs_inst, double* tp_db) {
    if (!p || !frame || !state || !meters) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    CK(cudaSetDevice(p->device));
    const int W = p->W;
    StreamCtx* c = stream_ctx(p);
    // staging layout (doubles): frame [W] | lufs, tp [2] | meters (5 floats in 4 doubles) | state [ST_STATE]
    const size_t n_d = (size_t)W + 2 + 4 + ST_STATE;
    int rc = c->ensure64(n_d * sizeof(double)); if (rc) return rc;
    double* h = c->h64; double* d = (double*)c->d64.p;
    memcpy(h, frame, (size_t)W * sizeof(double));
    size_t up = (size_t)W;
    if (!fresh) { memcpy(h + W + 6, state, ST_STATE * sizeof(double)); }
    CK(cudaMemcpyAsync(d, h, up * sizeof(double), cudaMemcpyHostToDevice, c->s));
    if (!fresh) CK(cudaMemcpyAsync(d + W + 6, h + W + 6, ST_STATE * sizeof(double), cudaMemcpyHostToDevice, c->s));
    {
        KweightArgs k;
        memset(&k, 0, sizeof k);
        k.x = d; k.x_is_f64 = 1; k.ch_stride = 0; k.frame_stride = W; k.frame_off0 = 0;
        k.n_ch = 1; k.n_frames = 1; k.first_frame = 0; k.frames_per_warp = 1;
        k.hann = nullptr; k.lufs_out = d + W; k.weighted_out = nullptr;
        fill_weighting(p, &k);
        p->launches++;
        rc = launch_kweight(k, c->s); if (rc) return rc;
        TruePeakArgs t;
        memset(&t, 0, sizeof t);
        t.x = d; t.x_is_f64 = 1; t.ch_stride = 0; t.frame_stride = W; t.frame_off0 = 0;
        t.n_ch = 1; t.n_frames = 1; t.first_frame = 0; t.rounds = 1;
        t.window = nullptr; t.twM = p->tw_meter.twM; t.rot = p->tp_rot;
        fill_truepeak_steps(&t);
        t.tp_out = d + W + 1;
        p->launches++;
        rc = launch_truepeak(t, c->s); if (rc) return rc;
        StatsArgs st;
        memset(&st, 0, sizeof st);
        st.lufs = d + W; st.tp = d + W + 1; st.n_ch = 1; st.n_frames = 1; st.first_frame = 0;
        st.gate = p->gate; st.out = (float*)(d + W + 2); st.fresh = fresh ? 1 : 0; st.state = d + W + 6;
        p->launches++;
        rc = launch_stats(st, c->s); if (rc) return rc;
    }
    CK(cudaMemcpyAsync(h + W, d + W, (6 + ST_STATE) * sizeof(double), cudaMemcpyDeviceToHost, c->s));
    CK(cudaStreamSynchronize(c->s));
    if (lufs_inst) *lufs_inst = h[W];
    if (tp_db) *tp_db = h[W + 1];
    memcpy(meters, h + W + 2, 5 * sizeof(float));
    memcpy(state, h + W + 6, ST_STATE * sizeof(double));
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// combine on caller-supplied magnitudes
// ------------------------------------------------------------------------------------------
extern "C" int omega4_combine(omega4_plan* p, void* stream, int mem, const float* const* magnitudes, int n_rows,
                              float* combined) {
    if (!p || !magnitudes || !combined || n_rows < 0) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_rows == 0) return OMEGA4_OK;
    CK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    CombineArgs c;
    memset(&c, 0, sizeof c);
    float* d_out = combined;
    if (mem == OMEGA4_MEM_HOST) {
        for (int r = 0; r < p->n_res; ++r)
            if (magnitudes[r]) {
                const size_t bytes = (size_t)n_rows * p->res[r].bins * sizeof(float);
                int rc = p->h_mag[r].ensure(bytes); if (rc) return rc;
                CK(cudaMemcpyAsync(p->h_mag[r].p, magnitudes[r], bytes, cudaMemcpyHostToDevice, s));
                c.mag[r] = (const float*)p->h_mag[r].p;
            }
        int rc = p->h_comb.ensure((size_t)n_rows * p->T * sizeof(float)); if (rc) return rc;
        d_out = (float*)p->h_comb.p;
    } else {
        for (int r = 0; r < p->n_res; ++r) c.mag[r] = magnitudes[r];
    }
    for (int r = 0; r < p->n_res; ++r) { c.bins[r] = p->res[r].bins; c.first_frame[r] = 0; c.weight[r] = p->res[r].weight; }
    c.n_hops = 0; c.n_rows = n_rows; c.T = p->T;
    c.csr_ptr = p->csr_ptr; c.csr_res = p->csr_res; c.csr_lo = p->csr_lo; c.csr_frac = p->csr_frac;
    c.out = d_out;
    const long long total = (long long)n_rows * p->T;
    p->launches++;
    combine_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(c);
    CK(cudaGetLastError());
    if (mem == OMEGA4_MEM_HOST) {
        CK(cudaMemcpyAsync(combined, d_out, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// meters on explicit frames / series
// ------------------------------------------------------------------------------------------
extern "C" int omega4_meter_frames(omega4_plan* p, void* stream, int mem, const double* frames, int n_frames,
                                   double* lufs_inst, double* tp_db, double* weighted) {
    if (!p || !frames || n_frames < 0) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_frames == 0) return OMEGA4_OK;
    CK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int W = p->W;
    const double* d_fr = frames; double* d_l = lufs_inst; double* d_t = tp_db; double* d_w = weighted;
    DevBuf tmp_w;
    if (mem == OMEGA4_MEM_HOST) {
        int rc = p->h_f64a.ensure((size_t)n_frames * W * sizeof(double)); if (rc) return rc;
        CK(cudaMemcpyAsync(p->h_f64a.p, frames, (size_t)n_frames * W * sizeof(double), cudaMemcpyHostToDevice, s));
        d_fr = (const double*)p->h_f64a.p;
        rc = p->h_f64b.ensure((size_t)n_frames * 2 * sizeof(double)); if (rc) return rc;
        d_l = (double*)p->h_f64b.p; d_t = d_l + n_frames;
        if (weighted) { rc = tmp_w.ensure((size_t)n_frames * W * sizeof(double)); if (rc) return rc; d_w = (double*)tmp_w.p; }
    } else if (((uintptr_t)frames & 15) != 0) {
        return fail(OMEGA4_ERR_INVALID, "frames must be 16-byte aligned");
    }
    int rc = OMEGA4_OK;
    if (lufs_inst || weighted) {
        if (!d_l || (mem == OMEGA4_MEM_DEVICE && !lufs_inst)) { rc = p->scratch_lufs.ensure((size_t)n_frames * sizeof(double)); if (rc) { tmp_w.release(); return rc; } d_l = (double*)p->scratch_lufs.p; }
        KweightArgs k;
        memset(&k, 0, sizeof k);
        k.x = d_fr; k.x_is_f64 = 1; k.ch_stride = 0; k.frame_stride = W; k.frame_off0 = 0;
        k.n_ch = 1; k.n_frames = n_frames; k.first_frame = 0; k.frames_per_warp = n_frames >= 64 ? 4 : 1;
        k.hann = nullptr; k.lufs_out = d_l; k.weighted_out = d_w;
        fill_weighting(p, &k);
        p->launches++;
        rc = launch_kweight(k, s);
        if (rc) { tmp_w.release(); return rc; }
    }
    if (tp_db) {
        TruePeakArgs t;
        memset(&t, 0, sizeof t);
        t.x = d_fr; t.x_is_f64 = 1; t.ch_stride = 0; t.frame_stride = W; t.frame_off0 = 0;
        t.n_ch = 1; t.n_frames = n_frames; t.first_frame = 0; t.rounds = default_rounds((n_frames + 1) / 2, 2);
        t.window = nullptr; t.twM = p->tw_meter.twM; t.rot = p->tp_rot;
        fill_truepeak_steps(&t);
        t.tp_out = d_t;
        p->launches++;
        rc = launch_truepeak(t, s);
        if (rc) { tmp_w.release(); return rc; }
    }
    if (mem == OMEGA4_MEM_HOST) {
        cudaError_t e = cudaSuccess;
        if (lufs_inst) e = cudaMemcpyAsync(lufs_inst, d_l, (size_t)n_frames * sizeof(double), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && tp_db) e = cudaMemcpyAsync(tp_db, d_t, (size_t)n_frames * sizeof(double), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && weighted) e = cudaMemcpyAsync(weighted, d_w, (size_t)n_frames * W * sizeof(double), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        tmp_w.release();
        if (e != cudaSuccess) return fail(OMEGA4_ERR_CUDA, std::string("meter_frames copy back failed: ") + cudaGetErrorString(e));
    }
    return OMEGA4_OK;
}

extern "C" int omega4_meter_stats(omega4_plan* p, void* stream, int mem, const double* lufs_inst, const double* tp_db,
                                  int n_ch, int n_frames, int first_frame, double* state, float* meters, int fresh) {
    if (!p || !lufs_inst || !tp_db || !meters || n_ch < 0 || n_frames < 0) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_ch == 0 || n_frames == 0) return OMEGA4_OK;
    CK(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    StatsArgs st;
    memset(&st, 0, sizeof st);
    const size_t rows = (size_t)n_ch * n_frames;
    st.n_ch = n_ch; st.n_frames = n_frames; st.first_frame = first_frame; st.gate = p->gate; st.fresh = fresh ? 1 : 0;
    if (mem == OMEGA4_MEM_HOST) {
        int rc = p->h_f64a.ensure(rows * 2 * sizeof(double)); if (rc) return rc;
        double* d = (double*)p->h_f64a.p;
        CK(cudaMemcpyAsync(d, lufs_inst, rows * sizeof(double), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(d + rows, tp_db, rows * sizeof(double), cudaMemcpyHostToDevice, s));
        st.lufs = d; st.tp = d + rows;
        rc = p->h_f64c.ensure((size_t)n_ch * ST_STATE * sizeof(double)); if (rc) return rc;
        st.state = (double*)p->h_f64c.p;
        if (state && !fresh) CK(cudaMemcpyAsync(st.state, state, (size_t)n_ch * ST_STATE * sizeof(double), cudaMemcpyHostToDevice, s));
        else st.fresh = 1;
        rc = p->h_meters.ensure(rows * 5 * sizeof(float)); if (rc) return rc;
        st.out = (float*)p->h_meters.p;
    } else {
        st.lufs = lufs_inst; st.tp = tp_db; st.out = meters;
        if (state) st.state = state;
        else { int rc = p->h_state.ensure((size_t)n_ch * ST_STATE * sizeof(double)); if (rc) return rc; st.state = (double*)p->h_state.p; st.fresh = 1; }
    }
    p->launches++;
    int rc = launch_stats(st, s);
    if (rc) return rc;
    if (mem == OMEGA4_MEM_HOST) {
        CK(cudaMemcpyAsync(meters, st.out, rows * 5 * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (state) CK(cudaMemcpyAsync(state, st.state, (size_t)n_ch * ST_STATE * sizeof(double), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// plan-less entry points
// ------------------------------------------------------------------------------------------
extern "C" int omega4_rfft_batch(int device, void* stream, int mem, const float* frames, int batch, int n,
                                 const float* window, float* magnitude, float* complex_out) {
    if (!frames || batch < 0 || (!magnitude && !complex_out)) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (!is_pow2(n) || n < 512 || n > 32768) return fail(OMEGA4_ERR_UNSUPPORTED, "fft size must be a power of two in 512 .. 32768");
    if (batch == 0) return OMEGA4_OK;
    if (omega4_device_count() == 0) return fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback");
    CK(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    const int log2m = ilog2(n) - 1, bins = n / 2 + 1;
    Twiddles tw;
    int rc = get_twiddles(device, log2m, &tw);
    if (rc) return rc;
    float* d_win = nullptr; float* d_in = nullptr; float* d_mag = nullptr; float2* d_c = nullptr;
    std::vector<void*> to_free;
    auto cleanup = [&]() { for (void* q : to_free) cudaFree(q); };
#define CKF(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { cleanup(); return fail(OMEGA4_ERR_CUDA, std::string(#expr " failed: ") + cudaGetErrorString(e__)); } } while (0)
    if (window) {
        CKF(cudaMalloc(&d_win, (size_t)n * sizeof(float))); to_free.push_back(d_win);
        CKF(cudaMemcpyAsync(d_win, window, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    if (mem == OMEGA4_MEM_HOST) {
        CKF(cudaMalloc(&d_in, (size_t)batch * n * sizeof(float))); to_free.push_back(d_in);
        CKF(cudaMemcpyAsync(d_in, frames, (size_t)batch * n * sizeof(float), cudaMemcpyHostToDevice, s));
        if (magnitude) { CKF(cudaMalloc(&d_mag, (size_t)batch * bins * sizeof(float))); to_free.push_back(d_mag); }
        if (complex_out) { CKF(cudaMalloc(&d_c, (size_t)batch * bins * sizeof(float2))); to_free.push_back(d_c); }
    } else {
        if (((uintptr_t)frames & 15) != 0) { cleanup(); return fail(OMEGA4_ERR_INVALID, "frames must be 16-byte aligned"); }
        d_in = const_cast<float*>(frames); d_mag = magnitude; d_c = reinterpret_cast<float2*>(complex_out);
    }
    MultiresArgs a;
    memset(&a, 0, sizeof a);
    a.x = d_in; a.ch_stride = 0; a.frame_stride = n; a.frame_off0 = 0;
    a.n_ch = 1; a.n_frames = batch; a.first_frame = 0;
    a.rounds = default_rounds(batch, (1 << log2m) >= 4096 ? 1 : 4096 >> log2m);
    a.window = d_win; a.binw = nullptr; a.twM = tw.twM; a.twN = tw.twN;
    a.mag_out = d_mag; a.cplx_out = d_c; a.comb_out = nullptr; a.T = 0; a.n_tb = 0; a.need_lo = 0; a.need_cnt = 0;
    rc = launch_multires(log2m, a, s);
    if (rc) { cleanup(); return rc; }
    if (mem == OMEGA4_MEM_HOST) {
        if (magnitude) CKF(cudaMemcpyAsync(magnitude, d_mag, (size_t)batch * bins * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (complex_out) CKF(cudaMemcpyAsync(complex_out, d_c, (size_t)batch * bins * sizeof(float2), cudaMemcpyDeviceToHost, s));
    }
    if (!to_free.empty()) CKF(cudaStreamSynchronize(s));
    cleanup();
#undef CKF
    return OMEGA4_OK;
}

extern "C" int omega4_band_map(int device, void* stream, int mem, const float* spectrum, int n_rows, int len,
                               const int* bands, int n_bars, const float* comp, float* bars_out, int db) {
    if (!spectrum || !bands || !bars_out || n_rows < 0 || len <= 0 || n_bars <= 0) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_rows == 0) return OMEGA4_OK;
    if (omega4_device_count() == 0) return fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback");
    CK(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    int n_valid = n_bars;
    for (int b = 0; b < n_bars; ++b) {
        if (bands[2 * b] < 0 || bands[2 * b + 1] < bands[2 * b]) return fail(OMEGA4_ERR_INVALID, "bad band table");
        if (bands[2 * b + 1] > len) { n_valid = b; break; }        // freq_mapper.py:188-189 `break`
    }
    std::vector<void*> to_free;
    auto cleanup = [&]() { for (void* q : to_free) cudaFree(q); };
#define CKF(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { cleanup(); return fail(OMEGA4_ERR_CUDA, std::string(#expr " failed: ") + cudaGetErrorString(e__)); } } while (0)
    int* d_bands = nullptr; float* d_comp = nullptr; const float* d_spec = spectrum; float* d_out = bars_out;
    CKF(cudaMalloc(&d_bands, (size_t)n_bars * 2 * sizeof(int))); to_free.push_back(d_bands);
    CKF(cudaMemcpyAsync(d_bands, bands, (size_t)n_bars * 2 * sizeof(int), cudaMemcpyHostToDevice, s));
    if (comp) {
        CKF(cudaMalloc(&d_comp, (size_t)len * sizeof(float))); to_free.push_back(d_comp);
        CKF(cudaMemcpyAsync(d_comp, comp, (size_t)len * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    if (mem == OMEGA4_MEM_HOST) {
        float* t = nullptr;
        CKF(cudaMalloc(&t, (size_t)n_rows * len * sizeof(float))); to_free.push_back(t);
        CKF(cudaMemcpyAsync(t, spectrum, (size_t)n_rows * len * sizeof(float), cudaMemcpyHostToDevice, s));
        d_spec = t;
        CKF(cudaMalloc(&d_out, (size_t)n_rows * n_bars * sizeof(float))); to_free.push_back(d_out);
    }
    const long long total = (long long)n_rows * n_bars;
    band_map_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(d_spec, n_rows, len, d_bands, n_bars, n_valid, d_comp, d_out, db);
    CKF(cudaGetLastError());
    if (mem == OMEGA4_MEM_HOST) CKF(cudaMemcpyAsync(bars_out, d_out, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, s));
    CKF(cudaStreamSynchronize(s));
    cleanup();
#undef CKF
    return OMEGA4_OK;
}

extern "C" int omega4_waterfall(int device, void* stream, int mem, const float* spectra, int n_ch, int n_rows, int len,
                                int lo, int hi, int db_form, int auto_gain, float gain_adjustment, float* state, int fresh,
                                float* db_out, float* norm_out, float* rowstat_out) {
    if (!spectra || n_ch < 0 || n_rows < 0 || len <= 0 || lo < 0 || hi <= lo || hi > len || (db_form != 0 && db_form != 1) ||
        (!db_out && !norm_out && !rowstat_out))
        return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_ch == 0 || n_rows == 0) return OMEGA4_OK;
    if ((long long)n_ch * n_rows > 2147483647LL) return fail(OMEGA4_ERR_INVALID, "too many rows for one waterfall call");
    if (omega4_device_count() == 0) return fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback");
    CK(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t rows = (size_t)n_ch * n_rows, n = (size_t)(hi - lo);
    std::vector<void*> to_free;
    auto cleanup = [&]() { for (void* q : to_free) cudaFree(q); };
#define CKF(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { cleanup(); return fail(OMEGA4_ERR_CUDA, std::string(#expr " failed: ") + cudaGetErrorString(e__)); } } while (0)
    WaterfallArgs a;
    memset(&a, 0, sizeof a);
    a.n_ch = n_ch; a.n_rows = n_rows; a.len = len; a.lo = lo; a.hi = hi; a.db_form = db_form; a.auto_gain = auto_gain ? 1 : 0;
    a.gain_adjustment = gain_adjustment;
    const size_t st_bytes = (size_t)n_ch * WF_STATE * sizeof(float);
    if (mem == OMEGA4_MEM_HOST) {
        float* t = nullptr;
        CKF(cudaMalloc(&t, rows * len * sizeof(float))); to_free.push_back(t);
        CKF(cudaMemcpyAsync(t, spectra, rows * len * sizeof(float), cudaMemcpyHostToDevice, s));
        a.spec = t;
        if (db_out) { CKF(cudaMalloc(&a.db_out, rows * n * sizeof(float))); to_free.push_back(a.db_out); }
        if (norm_out) { CKF(cudaMalloc(&a.norm_out, rows * n * sizeof(float))); to_free.push_back(a.norm_out); }
        if (state) {
            float* d_st = nullptr;
            CKF(cudaMalloc(&d_st, st_bytes)); to_free.push_back(d_st);
            if (!fresh) { CKF(cudaMemcpyAsync(d_st, state, st_bytes, cudaMemcpyHostToDevice, s)); a.state_in = d_st; }
            a.state_out = d_st;
        }
    } else if (mem == OMEGA4_MEM_DEVICE) {
        a.spec = spectra; a.db_out = db_out; a.norm_out = norm_out;
        a.state_in = (state && !fresh) ? state : nullptr; a.state_out = state;
    } else {
        return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");
    }
    if (mem == OMEGA4_MEM_DEVICE && rowstat_out) a.rowstat = rowstat_out;
    else { CKF(cudaMalloc(&a.rowstat, rows * 4 * sizeof(float))); to_free.push_back(a.rowstat); }
    waterfall_db_kernel<<<(unsigned)rows, 256, 0, s>>>(a);
    CKF(cudaGetLastError());
    waterfall_norm_kernel<<<(unsigned)rows, 256, 0, s>>>(a);
    CKF(cudaGetLastError());
    if (a.state_out) {
        waterfall_state_kernel<<<(unsigned)((n_ch + 127) / 128), 128, 0, s>>>(a);
        CKF(cudaGetLastError());
    }
    if (mem == OMEGA4_MEM_HOST) {
        if (db_out) CKF(cudaMemcpyAsync(db_out, a.db_out, rows * n * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (norm_out) CKF(cudaMemcpyAsync(norm_out, a.norm_out, rows * n * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (rowstat_out) CKF(cudaMemcpyAsync(rowstat_out, a.rowstat, rows * 4 * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (state) CKF(cudaMemcpyAsync(state, a.state_out, st_bytes, cudaMemcpyDeviceToHost, s));
    }
    if (!to_free.empty()) CKF(cudaStreamSynchronize(s));
    cleanup();
#undef CKF
    return OMEGA4_OK;
}

extern "C" int omega4_plan_set_gate_threshold(omega4_plan* p, double gate_threshold) {
    if (!p) return fail(OMEGA4_ERR_INVALID, "plan is NULL");
    if (!(gate_threshold == gate_threshold)) return fail(OMEGA4_ERR_INVALID, "gate threshold is NaN");
    p->gate = gate_threshold;
    return OMEGA4_OK;
}

extern "C" int omega4_bass_bars(int device, void* stream, int mem, const float* magnitudes, int n_ch, int n_frames,
                                int n_bins, const int* bar_bins, const float* comp, int n_bars, float* state,
                                float* bars_out) {
    if (!magnitudes || !bar_bins || !comp || !bars_out || n_ch < 0 || n_frames < 0 || n_bins <= 0 || n_bars <= 0 || n_bars > 128)
        return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_ch == 0 || n_frames == 0) return OMEGA4_OK;
    for (int b = 0; b < n_bars; ++b)
        if (bar_bins[2 * b] < 0 || bar_bins[2 * b + 1] < 0 || bar_bins[2 * b] + bar_bins[2 * b + 1] > n_bins)
            return fail(OMEGA4_ERR_INVALID, "bar bins out of range");
    if (omega4_device_count() == 0) return fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback");
    CK(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    std::vector<void*> to_free;
    auto cleanup = [&]() { for (void* q : to_free) cudaFree(q); };
#define CKF(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { cleanup(); return fail(OMEGA4_ERR_CUDA, std::string(#expr " failed: ") + cudaGetErrorString(e__)); } } while (0)
    int* d_bins = nullptr; float* d_comp = nullptr;
    CKF(cudaMalloc(&d_bins, (size_t)n_bars * 2 * sizeof(int))); to_free.push_back(d_bins);
    CKF(cudaMalloc(&d_comp, (size_t)n_bars * sizeof(float))); to_free.push_back(d_comp);
    CKF(cudaMemcpyAsync(d_bins, bar_bins, (size_t)n_bars * 2 * sizeof(int), cudaMemcpyHostToDevice, s));
    CKF(cudaMemcpyAsync(d_comp, comp, (size_t)n_bars * sizeof(float), cudaMemcpyHostToDevice, s));
    const float* d_mag = magnitudes; float* d_out = bars_out; float* d_state = state;
    const size_t rows = (size_t)n_ch * n_frames;
    if (mem == OMEGA4_MEM_HOST) {
        float* t = nullptr;
        CKF(cudaMalloc(&t, rows * n_bins * sizeof(float))); to_free.push_back(t);
        CKF(cudaMemcpyAsync(t, magnitudes, rows * n_bins * sizeof(float), cudaMemcpyHostToDevice, s));
        d_mag = t;
        CKF(cudaMalloc(&d_out, rows * n_bars * sizeof(float))); to_free.push_back(d_out);
        if (state) {
            CKF(cudaMalloc(&d_state, (size_t)n_ch * n_bars * sizeof(float))); to_free.push_back(d_state);
            CKF(cudaMemcpyAsync(d_state, state, (size_t)n_ch * n_bars * sizeof(float), cudaMemcpyHostToDevice, s));
        }
    } else if (mem != OMEGA4_MEM_DEVICE) {
        cleanup();
        return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");
    }
    bass_bars_kernel<<<(unsigned)((n_ch + 3) / 4), 128, 0, s>>>(d_mag, n_ch, n_frames, n_bins, d_bins, d_comp, n_bars, d_state, d_out);
    CKF(cudaGetLastError());
    if (mem == OMEGA4_MEM_HOST) {
        CKF(cudaMemcpyAsync(bars_out, d_out, rows * n_bars * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (state) CKF(cudaMemcpyAsync(state, d_state, (size_t)n_ch * n_bars * sizeof(float), cudaMemcpyDeviceToHost, s));
    }
    CKF(cudaStreamSynchronize(s));
    cleanup();
#undef CKF
    return OMEGA4_OK;
}

extern "C" int omega4_synth_fill(int device, void* stream, float* out_device, int n_streams, int n_channels,
                                 long long n_samples, long long row_stride, int first_stream, int sample_rate,
                                 long long clip_samples) {
    if (!out_device || n_streams < 0 || n_channels <= 0 || n_samples < 0 || row_stride < n_samples || sample_rate <= 0)
        return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_streams == 0 || n_samples == 0) return OMEGA4_OK;
    if (omega4_device_count() == 0) return fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback");
    CK(cudaSetDevice(device));
    const int rows = n_streams * n_channels;
    if (rows > 65535) return fail(OMEGA4_ERR_INVALID, "too many rows for one synth launch (max 65535)");
    const double clip_s = (double)(clip_samples > 0 ? clip_samples : n_samples) / sample_rate;
    dim3 grid((unsigned)((n_samples + 255) / 256), rows);
    synth_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out_device, rows, n_channels, n_samples, row_stride, first_stream,
                                                         (double)sample_rate, clip_s);
    CK(cudaGetLastError());
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// application post-processing: combined spectrum -> band_values (omega4_main.py:992-1056)
// ------------------------------------------------------------------------------------------
extern "C" omega4_bars* omega4_bars_create(const omega4_bars_desc* d, int device) {
    if (!d || !d->bands || d->spectrum_len < 2 || d->n_bars < 1 || d->percentile < 0 || d->percentile > 100) {
        fail(OMEGA4_ERR_INVALID, "bad bars descriptor"); return nullptr;
    }
    if (omega4_device_count() == 0) { fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback"); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { fail(OMEGA4_ERR_CUDA, "cudaSetDevice failed"); return nullptr; }
    omega4_bars* b = new omega4_bars();
    b->device = device; b->T = d->spectrum_len; b->scale = d->scale; b->normalize_max = d->normalize_max;
    int nv = 0;
    for (int i = 0; i < d->n_bars; ++i) {
        const int s = d->bands[2 * i], e = d->bands[2 * i + 1];
        if (s < 0 || e < s) { delete b; fail(OMEGA4_ERR_INVALID, "bad band table"); return nullptr; }
        if (e > d->spectrum_len) break;                            // omega4_main.py:1012-1013
        ++nv;
    }
    if (nv < 1 || nv > 2048) { delete b; fail(OMEGA4_ERR_UNSUPPORTED, "1..2048 bands must fit the spectrum"); return nullptr; }
    b->n_valid = nv;
    // np.percentile, method='linear': virtual index q/100 (n-1)
    const double vi = d->percentile / 100.0 * (d->spectrum_len - 1);
    b->p_lo = (int)floor(vi);
    if (b->p_lo > d->spectrum_len - 2) b->p_lo = d->spectrum_len - 2;
    b->p_frac = (float)(vi - b->p_lo);
    std::vector<float> sf(nv), sfc(nv);
    if (d->smooth) for (int i = 0; i < nv; ++i) { sf[i] = (float)d->smooth[i]; sfc[i] = (float)(1.0 - d->smooth[i]); }
    bool ok = upload((void**)&b->bands, d->bands, (size_t)nv * 2 * sizeof(int)) == OMEGA4_OK;
    if (ok && d->gain) ok = upload((void**)&b->gain, d->gain, (size_t)b->T * sizeof(float)) == OMEGA4_OK;
    if (ok && d->smooth) ok = upload((void**)&b->sf, sf.data(), nv * sizeof(float)) == OMEGA4_OK &&
                              upload((void**)&b->sfc, sfc.data(), nv * sizeof(float)) == OMEGA4_OK;
    if (!ok) { std::string keep = g_err; omega4_bars_destroy(b); g_err = keep; return nullptr; }
    return b;
}

extern "C" void omega4_bars_destroy(omega4_bars* b) {
    if (!b) return;
    cudaSetDevice(b->device);
    cudaFree(b->bands); cudaFree(b->gain); cudaFree(b->sf); cudaFree(b->sfc);
    b->h_spec.release(); b->h_out.release(); b->h_peak.release(); b->h_state.release(); b->state_in.release();
    cudaGetLastError();
    delete b;
}

extern "C" int omega4_bars_count(const omega4_bars* b) { return b ? b->n_valid : 0; }

extern "C" int omega4_bars_run(omega4_bars* b, void* stream, int mem, const float* spectrum, int n_ch, int n_hops,
                               float* state, int fresh, float* band_values, float* peak_values) {
    if (!b || !spectrum || !band_values || n_ch < 0 || n_hops < 0) return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (n_ch == 0 || n_hops == 0) return OMEGA4_OK;
    CK(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t rows = (size_t)n_ch * n_hops;
    const size_t st_bytes = (size_t)n_ch * (1 + b->n_valid) * sizeof(float);
    const float* d_spec = spectrum; float* d_out = band_values; float* d_peak = peak_values; float* d_state = state;
    const int is_fresh = (fresh || !state) ? 1 : 0;
    if (mem == OMEGA4_MEM_HOST) {
        int rc = b->h_spec.ensure(rows * b->T * sizeof(float)); if (rc) return rc;
        rc = b->h_out.ensure(rows * b->n_valid * sizeof(float)); if (rc) return rc;
        CK(cudaMemcpyAsync(b->h_spec.p, spectrum, rows * b->T * sizeof(float), cudaMemcpyHostToDevice, s));
        d_spec = (const float*)b->h_spec.p; d_out = (float*)b->h_out.p;
        if (peak_values) { rc = b->h_peak.ensure(rows * b->n_valid * sizeof(float)); if (rc) return rc; d_peak = (float*)b->h_peak.p; }
        if (state) {
            rc = b->h_state.ensure(st_bytes); if (rc) return rc;
            if (!is_fresh) CK(cudaMemcpyAsync(b->h_state.p, state, st_bytes, cudaMemcpyHostToDevice, s));
            d_state = (float*)b->h_state.p;
        }
    } else if (mem != OMEGA4_MEM_DEVICE) {
        return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");
    }
    {
        int rc = bars_launch(b, s, d_spec, n_ch, n_hops, d_state, is_fresh, d_out, d_peak, &b->state_in);
        if (rc) return rc;
    }
    if (mem == OMEGA4_MEM_HOST) {
        CK(cudaMemcpyAsync(band_values, d_out, rows * b->n_valid * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (peak_values) CK(cudaMemcpyAsync(peak_values, d_peak, rows * b->n_valid * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (state) CK(cudaMemcpyAsync(state, d_state, st_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// ITU-R BS.1770-4 program loudness / EBU Tech 3342 loudness range (extension outside reference parity)
// ------------------------------------------------------------------------------------------
struct omega4_loudness {
    int device = 0, fs = 0, C = 0, sub = 0;
    double coef[10] = {};          // shelf b0 b1 b2 a1 a2, high-pass b0 b1 b2 a1 a2
    double w[LOUD_MAX_CH] = {};
    long long launches = 0;
    DevBuf E, P, FS, Z;            // push scratch
    DevBuf h_x, h_state, h_mom, h_st, h_peak, h_out;   // OMEGA4_MEM_HOST staging
};

extern "C" omega4_loudness* omega4_loudness_create(const omega4_loudness_desc* d, int device) {
    if (!d || !d->ch_weights || !d->shelf_b || !d->shelf_a || !d->hp_b || !d->hp_a) {
        fail(OMEGA4_ERR_INVALID, "bad loudness descriptor"); return nullptr;
    }
    if (d->sample_rate <= 0 || d->sample_rate % 10 != 0 || d->sub != d->sample_rate / 10) {
        fail(OMEGA4_ERR_INVALID, "sample rate must be a positive multiple of 10 and sub = sample_rate / 10"); return nullptr;
    }
    if (d->channels < 1 || d->channels > LOUD_MAX_CH) {
        fail(OMEGA4_ERR_INVALID, "channels per stream must be 1 .. OMEGA4_LOUDNESS_MAX_CH"); return nullptr;
    }
    for (int c = 0; c < d->channels; ++c)
        if (!(d->ch_weights[c] >= 0.0) || !isfinite(d->ch_weights[c])) {
            fail(OMEGA4_ERR_INVALID, "channel weights must be finite and >= 0"); return nullptr;
        }
    const double* sec[4] = {d->shelf_b, d->shelf_a, d->hp_b, d->hp_a};
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 3; ++j)
            if (!isfinite(sec[i][j])) { fail(OMEGA4_ERR_INVALID, "K-weighting coefficients must be finite"); return nullptr; }
    if (d->shelf_a[0] != 1.0 || d->hp_a[0] != 1.0) { fail(OMEGA4_ERR_INVALID, "biquads must be normalised (a[0] = 1)"); return nullptr; }
    if (omega4_device_count() == 0) { fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback"); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { fail(OMEGA4_ERR_CUDA, "cudaSetDevice failed"); return nullptr; }
    omega4_loudness* h = new omega4_loudness();
    h->device = device; h->fs = d->sample_rate; h->C = d->channels; h->sub = d->sub;
    const double q[10] = {d->shelf_b[0], d->shelf_b[1], d->shelf_b[2], d->shelf_a[1], d->shelf_a[2],
                          d->hp_b[0], d->hp_b[1], d->hp_b[2], d->hp_a[1], d->hp_a[2]};
    memcpy(h->coef, q, sizeof q);
    for (int c = 0; c < d->channels; ++c) h->w[c] = d->ch_weights[c];
    return h;
}

extern "C" void omega4_loudness_destroy(omega4_loudness* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    for (DevBuf* b : {&h->E, &h->P, &h->FS, &h->Z, &h->h_x, &h->h_state, &h->h_mom, &h->h_st, &h->h_peak, &h->h_out})
        b->release();
    cudaGetLastError();
    delete h;
}

extern "C" int omega4_loudness_state_doubles(const omega4_loudness* h) { return h ? loud_state_doubles(h->C) : 0; }

extern "C" long long omega4_loudness_launches(const omega4_loudness* h) { return h ? h->launches : 0; }

extern "C" int omega4_loudness_push(omega4_loudness* h, void* stream, int mem, const float* samples, long long ch_stride,
                                    int n_streams, long long n_samples, double* state, int fresh, long long out_stride,
                                    float* momentary, float* short_term, float* sample_peak) {
    if (!h || !samples || !state || n_streams < 0 || n_samples < 0 || ch_stride < n_samples || out_stride < 0)
        return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (mem != OMEGA4_MEM_HOST && mem != OMEGA4_MEM_DEVICE)
        return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");
    if (n_streams == 0 || n_samples == 0) return OMEGA4_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int C = h->C, SD = loud_state_doubles(C);
    const long long rows = (long long)n_streams * C;
    const long long nsegb = n_samples / h->sub + 2;
    if (nsegb > 2147483647LL / 32 || rows * nsegb > 2147483647LL * 4)
        return fail(OMEGA4_ERR_INVALID, "push too large: split it into shorter tiles");
    LoudArgs a;
    memset(&a, 0, sizeof a);
    a.x = samples; a.ch_stride = ch_stride; a.n = n_samples; a.n_streams = n_streams; a.C = C; a.sub = h->sub;
    a.nsegb = (int)nsegb;
    a.sb0 = h->coef[0]; a.sb1 = h->coef[1]; a.sb2 = h->coef[2]; a.sa1 = h->coef[3]; a.sa2 = h->coef[4];
    a.hb0 = h->coef[5]; a.hb1 = h->coef[6]; a.hb2 = h->coef[7]; a.ha1 = h->coef[8]; a.ha2 = h->coef[9];
    for (int c = 0; c < C; ++c) a.w[c] = h->w[c];
    a.state = state; a.fresh = fresh ? 1 : 0;
    a.mom = momentary; a.st = short_term; a.out_stride = out_stride; a.peak_db = sample_peak;
    int rc;
    if ((rc = h->E.ensure((size_t)rows * nsegb * sizeof(double)))) return rc;
    if ((rc = h->P.ensure((size_t)rows * nsegb * sizeof(float)))) return rc;
    if ((rc = h->FS.ensure((size_t)rows * 4 * sizeof(double)))) return rc;
    if ((rc = h->Z.ensure((size_t)n_streams * nsegb * sizeof(double)))) return rc;
    a.E = (double*)h->E.p; a.P = (float*)h->P.p; a.FS = (double*)h->FS.p; a.Z = (double*)h->Z.p;
    long long ndone = 0;
    const size_t st_bytes = (size_t)n_streams * SD * sizeof(double);
    if (mem == OMEGA4_MEM_HOST) {
        // host state is readable here: T is common to the streams of one state array
        const long long T = fresh ? 0 : (long long)state[0];
        ndone = (T + n_samples) / h->sub - T / h->sub;
        if ((momentary || short_term) && out_stride < ndone) return fail(OMEGA4_ERR_INVALID, "out_stride below the step count");
        if ((rc = h->h_x.ensure((size_t)rows * n_samples * sizeof(float)))) return rc;
        if ((rc = h->h_state.ensure(st_bytes))) return rc;
        CK(cudaMemcpy2DAsync(h->h_x.p, n_samples * sizeof(float), samples, ch_stride * sizeof(float),
                             n_samples * sizeof(float), rows, cudaMemcpyHostToDevice, s));
        if (!fresh) CK(cudaMemcpyAsync(h->h_state.p, state, st_bytes, cudaMemcpyHostToDevice, s));
        a.x = (const float*)h->h_x.p; a.ch_stride = n_samples; a.state = (double*)h->h_state.p;
        a.out_stride = ndone;
        a.mom = a.st = nullptr; a.peak_db = nullptr;
        if (momentary && ndone) { if ((rc = h->h_mom.ensure((size_t)n_streams * ndone * sizeof(float)))) return rc; a.mom = (float*)h->h_mom.p; }
        if (short_term && ndone) { if ((rc = h->h_st.ensure((size_t)n_streams * ndone * sizeof(float)))) return rc; a.st = (float*)h->h_st.p; }
        if (sample_peak) { if ((rc = h->h_peak.ensure((size_t)rows * sizeof(float)))) return rc; a.peak_db = (float*)h->h_peak.p; }
    }
    const long long warps = (rows * ((nsegb + LOUD_GROUP - 1) / LOUD_GROUP) + 31) / 32;
    loudness_chain_kernel<<<(unsigned)((warps + LOUD_WARPS - 1) / LOUD_WARPS), LOUD_WARPS * 32, 0, s>>>(a);
    CK(cudaGetLastError());
    loudness_finalize_kernel<<<(unsigned)((n_streams + LOUD_WARPS - 1) / LOUD_WARPS), LOUD_WARPS * 32, 0, s>>>(a);
    CK(cudaGetLastError());
    h->launches += 2;
    if (mem == OMEGA4_MEM_HOST) {
        if (a.mom) CK(cudaMemcpy2DAsync(momentary, out_stride * sizeof(float), a.mom, ndone * sizeof(float),
                                        ndone * sizeof(float), n_streams, cudaMemcpyDeviceToHost, s));
        if (a.st) CK(cudaMemcpy2DAsync(short_term, out_stride * sizeof(float), a.st, ndone * sizeof(float),
                                       ndone * sizeof(float), n_streams, cudaMemcpyDeviceToHost, s));
        if (a.peak_db) CK(cudaMemcpyAsync(sample_peak, a.peak_db, (size_t)rows * sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(state, a.state, st_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return OMEGA4_OK;
}

extern "C" int omega4_loudness_summary(omega4_loudness* h, void* stream, int mem, const float* momentary,
                                       const float* short_term, int n_streams, int n_steps, long long stride, float* out) {
    if (!h || !momentary || !short_term || !out || n_streams < 0 || n_steps < 0 || stride < n_steps)
        return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (mem != OMEGA4_MEM_HOST && mem != OMEGA4_MEM_DEVICE)
        return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");
    if (n_streams == 0) return OMEGA4_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const float* m = momentary; const float* st = short_term; float* o = out;
    long long ld = stride;
    if (mem == OMEGA4_MEM_HOST) {
        const size_t bytes = (size_t)n_streams * (n_steps > 0 ? n_steps : 1) * sizeof(float);
        int rc;
        if ((rc = h->h_mom.ensure(bytes)) || (rc = h->h_st.ensure(bytes)) || (rc = h->h_out.ensure((size_t)n_streams * 4 * sizeof(float))))
            return rc;
        if (n_steps > 0) {
            CK(cudaMemcpy2DAsync(h->h_mom.p, n_steps * sizeof(float), momentary, stride * sizeof(float),
                                 n_steps * sizeof(float), n_streams, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpy2DAsync(h->h_st.p, n_steps * sizeof(float), short_term, stride * sizeof(float),
                                 n_steps * sizeof(float), n_streams, cudaMemcpyHostToDevice, s));
        }
        m = (const float*)h->h_mom.p; st = (const float*)h->h_st.p; o = (float*)h->h_out.p; ld = n_steps;
    }
    loudness_summary_kernel<<<(unsigned)n_streams, LOUD_SUM_THREADS, 0, s>>>(m, st, ld, n_steps, o);
    CK(cudaGetLastError());
    h->launches += 1;
    if (mem == OMEGA4_MEM_HOST) {
        CK(cudaMemcpyAsync(out, o, (size_t)n_streams * 4 * sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return OMEGA4_OK;
}

// ------------------------------------------------------------------------------------------
// One-third-octave band levels per channel (extension outside reference parity)
// ------------------------------------------------------------------------------------------
struct omega4_octave {
    int device = 0, fs = 0, nb = 0, sub = 0;
    long long launches = 0;
    DevBuf coef;                                   // [32][OCT_COEF] doubles
    DevBuf h_x, h_state, h_levels, h_leq, h_lmax;  // OMEGA4_MEM_HOST staging
};

// zeros at z = 1 and z = -1 of a numerator g [1, -2, 1], g [1, 2, 1] or g [1, 0, -1]; false for anything else
static bool oct_zero_pair(const double* b, int* plus, int* minus) {
    if (!(b[0] != 0.0) || !isfinite(b[0])) return false;
    if (b[1] == -2.0 * b[0] && b[2] == b[0]) { *plus += 2; return true; }
    if (b[1] == 2.0 * b[0] && b[2] == b[0]) { *minus += 2; return true; }
    if (b[1] == 0.0 && b[2] == -b[0]) { *plus += 1; *minus += 1; return true; }
    return false;
}

extern "C" omega4_octave* omega4_octave_create(const omega4_octave_desc* d, int device) {
    if (!d || !d->sos) { fail(OMEGA4_ERR_INVALID, "bad octave descriptor"); return nullptr; }
    if (d->sample_rate < 8000 || d->sample_rate > 192000 || d->sample_rate % 10 != 0 || d->sub != d->sample_rate / 10) {
        fail(OMEGA4_ERR_INVALID, "sample rate must be a multiple of 10 in [8000, 192000] and sub = sample_rate / 10");
        return nullptr;
    }
    if (d->n_bands < 1 || d->n_bands > OCT_MAX_BANDS) {
        fail(OMEGA4_ERR_INVALID, "n_bands must be 1 .. OMEGA4_OCTAVE_MAX_BANDS"); return nullptr;
    }
    double table[32 * OCT_COEF] = {};
    for (int b = 0; b < d->n_bands; ++b) {
        int plus = 0, minus = 0;
        double g = 1.0;
        for (int k = 0; k < 3; ++k) {
            const double* s = d->sos + (b * 3 + k) * 6;
            if (!oct_zero_pair(s, &plus, &minus)) {
                fail(OMEGA4_ERR_INVALID, "octave section numerators must be g [1, -2, 1], g [1, 2, 1] or g [1, 0, -1]");
                return nullptr;
            }
            const double a1 = s[4], a2 = s[5];
            if (s[3] != 1.0 || !isfinite(a1) || !isfinite(a2) || !(fabs(a2) < 1.0) || !(fabs(a1) < 1.0 + a2)) {
                fail(OMEGA4_ERR_INVALID, "octave sections must be normalised (a0 = 1) with poles inside the unit circle");
                return nullptr;
            }
            g *= s[0];
            table[b * OCT_COEF + 2 * k] = -a1;
            table[b * OCT_COEF + 2 * k + 1] = -a2;
        }
        if (plus != 3 || minus != 3) {
            fail(OMEGA4_ERR_INVALID, "each octave band needs three zeros at z = 1 and three at z = -1"); return nullptr;
        }
        table[b * OCT_COEF + 6] = 2.0 * g * g / d->sub;
        table[b * OCT_COEF + 7] = 2.0 * g * g;
    }
    table[d->n_bands * OCT_COEF + 6] = 2.0 / d->sub;      // the overall column: no filter, unit gain
    table[d->n_bands * OCT_COEF + 7] = 2.0;
    if (omega4_device_count() == 0) { fail(OMEGA4_ERR_NO_DEVICE, "no CUDA device visible: libomega4_cuda has no CPU fallback"); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { fail(OMEGA4_ERR_CUDA, "cudaSetDevice failed"); return nullptr; }
    omega4_octave* h = new omega4_octave();
    h->device = device; h->fs = d->sample_rate; h->nb = d->n_bands; h->sub = d->sub;
    const int rc = h->coef.ensure(sizeof table);          // sets the error message itself when it fails
    if (rc != OMEGA4_OK || cudaMemcpy(h->coef.p, table, sizeof table, cudaMemcpyHostToDevice) != cudaSuccess) {
        if (rc == OMEGA4_OK) fail(OMEGA4_ERR_CUDA, "copying the octave coefficients to the device failed");
        omega4_octave_destroy(h);
        return nullptr;
    }
    return h;
}

extern "C" void omega4_octave_destroy(omega4_octave* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    for (DevBuf* b : {&h->coef, &h->h_x, &h->h_state, &h->h_levels, &h->h_leq, &h->h_lmax}) b->release();
    cudaGetLastError();
    delete h;
}

extern "C" int omega4_octave_state_doubles(const omega4_octave* h) { return h ? oct_state_doubles(h->nb) : 0; }

extern "C" long long omega4_octave_launches(const omega4_octave* h) { return h ? h->launches : 0; }

extern "C" int omega4_octave_push(omega4_octave* h, void* stream, int mem, const float* samples, long long ch_stride,
                                  int n_rows, long long n_samples, double* state, int fresh, long long out_stride,
                                  float* levels, float* leq, float* lmax) {
    if (!h || !samples || !state || n_rows < 0 || n_samples < 0 || ch_stride < n_samples || out_stride < 0)
        return fail(OMEGA4_ERR_INVALID, "bad arguments");
    if (mem != OMEGA4_MEM_HOST && mem != OMEGA4_MEM_DEVICE)
        return fail(OMEGA4_ERR_INVALID, "mem must be OMEGA4_MEM_HOST or OMEGA4_MEM_DEVICE");
    if (((uintptr_t)samples & 3) || ((uintptr_t)state & 7) || ((uintptr_t)levels & 3) || ((uintptr_t)leq & 3) ||
        ((uintptr_t)lmax & 3))
        return fail(OMEGA4_ERR_INVALID, "samples, levels, leq and lmax must be float-aligned and state double-aligned");
    if (n_rows == 0 || n_samples == 0) return OMEGA4_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int ncol = h->nb + 1, SD = oct_state_doubles(h->nb);
    OctArgs a;
    memset(&a, 0, sizeof a);
    a.x = samples; a.ch_stride = ch_stride; a.n = n_samples; a.n_rows = n_rows; a.nb = h->nb; a.sub = h->sub;
    a.coef = (const double*)h->coef.p;
    a.state = state; a.fresh = fresh ? 1 : 0;
    a.levels = levels; a.out_stride = out_stride; a.leq = leq; a.lmax = lmax;
    long long ndone = 0;
    const size_t st_bytes = (size_t)n_rows * SD * sizeof(double);
    const size_t col_bytes = (size_t)n_rows * ncol * sizeof(float);
    int rc;
    if (mem == OMEGA4_MEM_HOST) {
        // host state is readable here: T is common to the rows of one state array
        const long long T = fresh ? 0 : (long long)state[0];
        ndone = (T + n_samples) / h->sub - T / h->sub;
        if (levels && out_stride < ndone) return fail(OMEGA4_ERR_INVALID, "out_stride below the block count of this push");
        if ((rc = h->h_x.ensure((size_t)n_rows * n_samples * sizeof(float)))) return rc;
        if ((rc = h->h_state.ensure(st_bytes))) return rc;
        CK(cudaMemcpy2DAsync(h->h_x.p, n_samples * sizeof(float), samples, ch_stride * sizeof(float),
                             n_samples * sizeof(float), n_rows, cudaMemcpyHostToDevice, s));
        if (!fresh) CK(cudaMemcpyAsync(h->h_state.p, state, st_bytes, cudaMemcpyHostToDevice, s));
        a.x = (const float*)h->h_x.p; a.ch_stride = n_samples; a.state = (double*)h->h_state.p;
        a.levels = nullptr; a.out_stride = ndone; a.leq = a.lmax = nullptr;
        if (levels && ndone) {
            if ((rc = h->h_levels.ensure((size_t)n_rows * ndone * ncol * sizeof(float)))) return rc;
            a.levels = (float*)h->h_levels.p;
        }
        if (leq) { if ((rc = h->h_leq.ensure(col_bytes))) return rc; a.leq = (float*)h->h_leq.p; }
        if (lmax) { if ((rc = h->h_lmax.ensure(col_bytes))) return rc; a.lmax = (float*)h->h_lmax.p; }
    }
    octave_kernel<<<(unsigned)((n_rows + OCT_WARPS - 1) / OCT_WARPS), OCT_WARPS * 32, 0, s>>>(a);
    CK(cudaGetLastError());
    h->launches += 1;
    if (mem == OMEGA4_MEM_HOST) {
        if (a.levels) CK(cudaMemcpy2DAsync(levels, out_stride * ncol * sizeof(float), a.levels, ndone * ncol * sizeof(float),
                                           ndone * ncol * sizeof(float), n_rows, cudaMemcpyDeviceToHost, s));
        if (a.leq) CK(cudaMemcpyAsync(leq, a.leq, col_bytes, cudaMemcpyDeviceToHost, s));
        if (a.lmax) CK(cudaMemcpyAsync(lmax, a.lmax, col_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(state, a.state, st_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return OMEGA4_OK;
}
