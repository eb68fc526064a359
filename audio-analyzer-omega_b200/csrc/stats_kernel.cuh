// stats_kernel.cuh -- the deque statistics of ProfessionalMetering.calculate_lufs.
//
// Replaces omega4/panels/professional_meters.py:248-279 for a series of per-frame values:
//   momentary  = mean of the last 24 instantaneous-LUFS values (dB domain, -100 entries included)
//   short_term = mean of the last 180
//   integrated = mean of the values > -70 among the last 3600, else -100
//   range      = P95 - P10 (numpy 'linear' percentile) of those gated values, else 0
//   true_peak  = max of the last 60 per-frame true peaks
// One CTA per channel walks the hops in order (the only sequential dependency of the whole
// path).  The window of the last 3600 values and a SORTED copy of its gated members live in
// shared memory; every hop removes the expiring value and inserts the new one by a parallel
// shift, so the exact order statistics numpy would compute are read directly.  State (the
// window, the peak window, the current outputs) is carried in global memory between calls so
// long streams can be processed in time tiles and the streaming shim can push one hop at a time.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

namespace o4 {

constexpr int ST_M = 24;       // int(0.4 * 60)
constexpr int ST_S = 180;      // int(3.0 * 60)
constexpr int ST_I = 3600;     // int(60 * 60)
constexpr int ST_P = 60;       // int(1.0 * 60)
constexpr int ST_SORT = 4096;  // padded sort size
constexpr int ST_THREADS = 32;     // one warp per channel
// per-channel state, in doubles: [0] n_hist, [1] n_tp, [2..6] current outputs, [8 .. 8+3600) window
// (oldest first), [8+3600 .. 8+3600+60) peak window (oldest first)
constexpr int ST_STATE = 8 + ST_I + ST_P;

struct StatsArgs {
    const double* lufs;        // [n_ch][n_frames]
    const double* tp;          // [n_ch][n_frames]
    int n_ch;
    int n_frames;
    int first_frame;           // hops before this do not push (no meter frame yet)
    double gate;               // -70
    double* state;             // [n_ch][ST_STATE], zero-initialised = fresh meters
    float* out;                // [n_ch][n_frames][5]  M, S, I, LRA, TP
    int fresh;                 // 1: ignore state contents on entry (treat as new meters)
};

__device__ __forceinline__ double st_percentile(const double* s, int n, double q) {
    // numpy.percentile(..., method='linear') on an ascending array of n >= 1 values
    double vi = (double)n * q + (1.0 + q * (1.0 - 1.0 - 1.0)) - 1.0;
    if (vi < 0.0) vi = 0.0;
    if (vi > (double)(n - 1)) vi = (double)(n - 1);
    double fl = floor(vi);
    int lo = (int)fl;
    int hi = lo + 1 < n ? lo + 1 : n - 1;
    double t = vi - fl;
    double av = s[lo], bv = s[hi];
    double d = bv - av;
    return (t >= 0.5) ? (bv - d * (1.0 - t)) : (av + d * t);
}

// first index i in [0, n) with s[i] >= v (n if none), found by one warp with a 32-ary search
__device__ __forceinline__ int warp_lower_bound(const float* s, int n, float v, int lane) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int step = (hi - lo + 31) >> 5;
        const int idx = lo + lane * step;
        const bool less = (idx < hi) && (s[idx] < v);
        const int c = __popc(__ballot_sync(0xffffffffu, less));
        if (step == 1) return lo + c;
        if (c == 0) return lo;
        const int nhi = min(hi, lo + c * step);
        lo = lo + (c - 1) * step + 1;
        hi = nhi;
    }
    return lo;
}

__device__ __forceinline__ double st_percentile_f(const float* s, int n, double q) {
    double vi = (double)n * q + (1.0 + q * (1.0 - 1.0 - 1.0)) - 1.0;
    if (vi < 0.0) vi = 0.0;
    if (vi > (double)(n - 1)) vi = (double)(n - 1);
    const double fl = floor(vi);
    const int lo = (int)fl;
    const int hi = lo + 1 < n ? lo + 1 : n - 1;
    const double t = vi - fl;
    const double av = (double)s[lo], bv = (double)s[hi];
    const double d = bv - av;
    return (t >= 0.5) ? (bv - d * (1.0 - t)) : (av + d * t);
}

// ONE WARP PER CHANNEL, no block barriers.  The per-frame values are rounded to float32 for the sorted copy and
// the sums (the outputs are float32; 4e-6 LU), and every sum adds and subtracts exactly those rounded values in
// double, so nothing drifts.  Gate membership is decided on the unrounded double against the double gate, as the
// reference does: a value in (-70, -70 + 3.8e-6) rounds to -70.0f but is a member.  Shared memory per channel:
// the sorted gated copy and the ring of the last 60 peaks only -- the window itself is never kept on chip: the value that expires from the 3600 / 180 / 24
// windows at hop k is the value pushed that many hops earlier, i.e. an element of the input series (or of
// the carried state), fetched one 32-hop slice ahead with the new values.  14.7 KB per channel -> 15 channels
// per SM: BASELINE's 2048 channels are resident in ONE wave (the kernel is a latency-bound sequential walk,
// its duration is hops x per-hop latency x waves; with the ring on chip it needed 31 KB and two waves, and
// squeezed the FFT kernels it overlaps out of shared memory).  CARRIED = state from an earlier call has to be
// sorted once: 4096 slots for the bitonic network (16.6 KB).
template <bool CARRIED>
constexpr int stw_smem() { return ((CARRIED ? ST_SORT : ST_I) + 64) * (int)sizeof(float); }

template <bool CARRIED>
__global__ void __launch_bounds__(32)
stats_kernel(const __grid_constant__ StatsArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* srt = reinterpret_cast<float*>(smem_raw);          // sorted gated values
    float* pkw = srt + (CARRIED ? ST_SORT : ST_I);            // ring of the last 60 peaks

    const int ch = blockIdx.x;
    const int lane = threadIdx.x;
    double* st = a.state + (size_t)ch * ST_STATE;
    const double* lufs = a.lufs + (size_t)ch * a.n_frames;
    const double* tps = a.tp + (size_t)ch * a.n_frames;

    int n_hist = 0, n_tp = 0;
    double cur[5] = {-100.0, -100.0, -100.0, 0.0, -100.0};
    if (CARRIED && !a.fresh) {
        // counts of a state vector the library did not write itself are clamped: they index shared memory
        n_hist = min(max((int)st[0], 0), ST_I);
        n_tp = min(max((int)st[1], 0), ST_P);
        if (n_hist > 0 || n_tp > 0 || st[7] != 0.0) {
#pragma unroll
            for (int i = 0; i < 5; ++i) cur[i] = st[2 + i];
        }
    }
    const int n0 = n_hist;                                    // carried window length (oldest first in st[8 ..])
    const double* win0 = st + 8;
    if (CARRIED) for (int i = lane; i < n_tp; i += 32) pkw[i] = (float)st[8 + ST_I + i];
    __syncwarp();
    // all lanes keep the same (uniform) bookkeeping
    int pk_head = 0, ns = 0, cnt_m = 0, cnt_s = 0;
    double sum_i = 0.0, sum_m = 0.0, sum_s = 0.0, inv_m = 1.0, inv_s = 1.0, inv_ns = 0.0;
    float tp_max = -CUDART_INF_F;
    if (CARRIED && (n_hist > 0 || n_tp > 0)) {                // carried state: rebuild the derived structures
        for (int i = lane; i < ST_SORT; i += 32) {
            const double v = (i < n_hist) ? win0[i] : 0.0;
            srt[i] = (i < n_hist && v > a.gate) ? (float)v : CUDART_INF_F;   // non-gated entries sort to the end
        }
        __syncwarp();
        for (int k = 2; k <= ST_SORT; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = lane; i < ST_SORT; i += 32) {
                    int ixj = i ^ j;
                    if (ixj > i) {
                        float x = srt[i], y = srt[ixj];
                        bool up = ((i & k) == 0);
                        if ((x > y) == up) { srt[i] = y; srt[ixj] = x; }
                    }
                }
                __syncwarp();
            }
        }
        double si = 0.0; int c = 0;
        for (int i = lane; i < n_hist; i += 32) { const double v = win0[i]; if (v > a.gate) { ++c; si += (double)(float)v; } }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { c += __shfl_xor_sync(0xffffffffu, c, o); si += __shfl_xor_sync(0xffffffffu, si, o); }
        ns = c; sum_i = si;
        cnt_m = n_hist < ST_M ? n_hist : ST_M;
        cnt_s = n_hist < ST_S ? n_hist : ST_S;
        for (int i = n_hist - cnt_m; i < n_hist; ++i) sum_m += (double)(float)win0[i];
        for (int i = n_hist - cnt_s; i < n_hist; ++i) sum_s += (double)(float)win0[i];
        if (cnt_m > 0) inv_m = 1.0 / (double)cnt_m;
        if (cnt_s > 0) inv_s = 1.0 / (double)cnt_s;
        if (ns > 0) inv_ns = 1.0 / (double)ns;
        float m = -CUDART_INF_F;
        for (int i = lane; i < n_tp; i += 32) m = fmaxf(m, pkw[i]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        tp_max = m;
    }
    // hops before the first meter frame keep the current outputs
    const int kbeg = a.first_frame < a.n_frames ? a.first_frame : a.n_frames;
    for (int k = lane; k < kbeg; k += 32) {
        float* orow = a.out + ((size_t)ch * a.n_frames + k) * 5;
#pragma unroll
        for (int i = 0; i < 5; ++i) orow[i] = (float)cur[i];
    }

    // the value pushed D pushes before push p of this call: an element of the series, or of the carried window
    auto pushed_before = [&](int p, int D) -> double {
        const int q = p - D;
        if (q >= 0) return lufs[kbeg + q];
        const int c = n0 + q;
        return (CARRIED && c >= 0) ? win0[c] : 0.0;
    };
    float my_l = 0.f, my_t = 0.f, my_oi = 0.f, my_os = 0.f, my_om = 0.f;   // lane i holds hop kb + i of the current 32-hop slice
    unsigned in_new = 0u;                                     // bit i: gate membership of the new value of hop kb + i
    for (int k = kbeg; k < a.n_frames; ++k) {
        const int kk = (k - kbeg) & 31;
        if (kk == 0) {
            const int idx = k + lane;
            const bool ok = idx < a.n_frames;
            const double l = ok ? lufs[idx] : 0.0;
            const double oi = ok ? pushed_before(idx - kbeg, ST_I) : 0.0;  // leaves the 3600 window at this hop
            my_l = (float)l;
            my_t = ok ? (float)tps[idx] : 0.f;
            my_oi = (oi > a.gate) ? (float)oi : CUDART_NAN_F;              // NaN: not a gated member
            my_os = ok ? (float)pushed_before(idx - kbeg, ST_S) : 0.f;     // leaves the 180 window
            my_om = ok ? (float)pushed_before(idx - kbeg, ST_M) : 0.f;     // leaves the 24 window
            in_new = __ballot_sync(0xffffffffu, ok && l > a.gate);
        }
        const float nv = __shfl_sync(0xffffffffu, my_l, kk);
        const float ntp = __shfl_sync(0xffffffffu, my_t, kk);
        const float ov_i = __shfl_sync(0xffffffffu, my_oi, kk);
        const float ov_s = __shfl_sync(0xffffffffu, my_os, kk);
        const float ov_m = __shfl_sync(0xffffffffu, my_om, kk);
        // ---- expiring value, positions in the sorted gated array
        const bool has_old = (n_hist == ST_I);
        const float ov = has_old ? ov_i : 0.f;
        const bool rem = has_old && !isnan(ov);
        const bool ins = (in_new >> kk) & 1u;
        const int prem = rem ? warp_lower_bound(srt, ns, ov, lane) : -1;
        const int pins = ins ? warp_lower_bound(srt, ns, nv, lane) : -1;   // position in the pre-removal array
        // ---- shift: remove old index prem, insert before old index pins
        int lo = ns, hi = -1;
        if (prem >= 0 && pins >= 0) {
            if (pins > prem) { lo = prem + 1; hi = pins - 1; }        // shift left by one
            else { lo = pins; hi = prem - 1; }                        // shift right by one
        } else if (prem >= 0) { lo = prem + 1; hi = ns - 1; }
        else if (pins >= 0) { lo = pins; hi = ns - 1; }
        const bool left = (prem >= 0 && (pins < 0 || pins > prem));
        if (hi >= lo) {
            constexpr int SB = 8;                                 // elements per lane and batch
            if (left) {                                       // ascending batches of 256: read, sync, write one lower
                for (int base = lo; base <= hi; base += 32 * SB) {
                    float tb[SB];
#pragma unroll
                    for (int j = 0; j < SB; ++j) { int idx = base + lane + 32 * j; if (idx <= hi) tb[j] = srt[idx]; }
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < SB; ++j) { int idx = base + lane + 32 * j; if (idx <= hi) srt[idx - 1] = tb[j]; }
                }
            } else {                                          // descending batches: read, sync, write one higher
                for (int top = hi; top >= lo; top -= 32 * SB) {
                    float tb[SB];
#pragma unroll
                    for (int j = 0; j < SB; ++j) { int idx = top - lane - 32 * j; if (idx >= lo) tb[j] = srt[idx]; }
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < SB; ++j) { int idx = top - lane - 32 * j; if (idx >= lo) srt[idx + 1] = tb[j]; }
                }
            }
        }
        __syncwarp();
        // ---- uniform bookkeeping + single-lane stores
        if (!has_old) ++n_hist;
        const int ns_new = ns + (ins ? 1 : 0) - (rem ? 1 : 0);
        if (rem) sum_i -= (double)ov;
        if (ins) sum_i += (double)nv;
        if (ns_new != ns) inv_ns = ns_new > 0 ? 1.0 / (double)ns_new : 0.0;
        ns = ns_new;
        if (ns == 0) sum_i = 0.0;
        sum_m += (double)nv;
        if (cnt_m == ST_M) sum_m -= (double)ov_m;
        else { ++cnt_m; inv_m = 1.0 / (double)cnt_m; }
        sum_s += (double)nv;
        if (cnt_s == ST_S) sum_s -= (double)ov_s;
        else { ++cnt_s; inv_s = 1.0 / (double)cnt_s; }
        int pslot;
        float otp = -CUDART_INF_F;
        if (n_tp == ST_P) { pslot = pk_head; otp = pkw[pk_head]; pk_head = (pk_head + 1 == ST_P) ? 0 : pk_head + 1; }
        else { pslot = n_tp; ++n_tp; }
        __syncwarp();                                         // every lane has read pkw[pk_head]
        if (lane == 0) {
            if (ins) srt[pins - ((prem >= 0 && pins > prem) ? 1 : 0)] = nv;
            pkw[pslot] = ntp;
        }
        __syncwarp();
        // sliding maximum of the last 60 peaks: rescan only when the expiring value was the maximum
        if (ntp >= tp_max) tp_max = ntp;
        else if (otp >= tp_max) {
            float m = -CUDART_INF_F;
            for (int i = lane; i < n_tp; i += 32) m = fmaxf(m, pkw[i]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            tp_max = m;
        }
        // ---- outputs
        double pv = (ns > 0 && lane < 2) ? st_percentile_f(srt, ns, lane == 0 ? 0.95 : 0.10) : 0.0;
        const double p10 = __shfl_sync(0xffffffffu, pv, 1);
        cur[0] = sum_m * inv_m;
        cur[1] = sum_s * inv_s;
        cur[2] = (ns > 0) ? sum_i * inv_ns : -100.0;
        cur[3] = (ns > 0) ? __shfl_sync(0xffffffffu, pv, 0) - p10 : 0.0;
        cur[4] = (double)tp_max;
        if (lane == 0) {
            float* orow = a.out + ((size_t)ch * a.n_frames + k) * 5;
            orow[0] = (float)cur[0]; orow[1] = (float)cur[1]; orow[2] = (float)cur[2];
            orow[3] = (float)cur[3]; orow[4] = (float)cur[4];
        }
    }
    __syncwarp();
    // ---- write state back (chronological order): the last n_hist entries of (carried window ++ this call's pushes).
    // In place: entry i comes from combined index c = i + shift >= i, so ascending 32-wide batches never read a
    // slot an earlier batch has overwritten.
    {
        const int P = a.n_frames - kbeg;                      // pushes of this call
        const int shift = n0 + P - n_hist;
        for (int b0 = 0; b0 < n_hist; b0 += 32) {
            const int i = b0 + lane;
            double v = 0.0;
            if (i < n_hist) {
                const int c = i + shift;
                v = (c < n0) ? win0[c] : lufs[kbeg + c - n0];     // unrounded: a later call decides membership on it
            }
            __syncwarp();
            if (i < n_hist) st[8 + i] = v;
        }
    }
    {
        float pv2[2] = {0.f, 0.f};                            // the peak ring has 60 entries: two per lane, read before any store
#pragma unroll
        for (int j = 0; j < 2; ++j) { const int i = lane + 32 * j; if (i < n_tp) pv2[j] = pkw[(n_tp == ST_P) ? (pk_head + i) % ST_P : i]; }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 2; ++j) { const int i = lane + 32 * j; if (i < n_tp) st[8 + ST_I + i] = (double)pv2[j]; }
    }
    if (lane == 0) {
        st[0] = (double)n_hist; st[1] = (double)n_tp; st[7] = 1.0;
        st[2] = cur[0]; st[3] = cur[1]; st[4] = cur[2]; st[5] = cur[3]; st[6] = cur[4];
    }
}


// ---------------------------------------------------------------------------------------------
// One frame per call on carried state (the streaming shim: ProfessionalMetering.calculate_lufs once per application
// frame).  The walking kernel above would rebuild the sorted gated window with ONE warp (a 4096-element bitonic
// network, ~0.3 ms) to push a single value; here a 256-thread CTA per channel sorts the gated values of the new window
// with block-wide steps (sort size = next power of two above the window length) and evaluates the statistics directly.
// The per-frame values are rounded to float32 and summed in double exactly as above (those sums are exact, so the
// order does not matter), and membership is decided on the unrounded values: the outputs are bit-identical to the
// walking kernel's.  The window is kept in double for that (44.5 KB of static shared memory).
// ---------------------------------------------------------------------------------------------
constexpr int ST_P1_THREADS = 256;

__global__ void __launch_bounds__(ST_P1_THREADS)
stats_push1_kernel(const __grid_constant__ StatsArgs a) {
    __shared__ double win[ST_I];                             // the new window, oldest first, unrounded
    __shared__ float srt[ST_SORT];
    __shared__ float pk[ST_P];
    __shared__ double red_d[ST_P1_THREADS / 32];
    __shared__ int red_i[ST_P1_THREADS / 32];
    const int ch = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* st = a.state + (size_t)ch * ST_STATE;
    const int n0 = min(max((int)st[0], 0), ST_I), p0 = min(max((int)st[1], 0), ST_P);
    const double nv = a.lufs[ch];
    const float ntp = (float)a.tp[ch];
    const int drop = (n0 == ST_I) ? 1 : 0, n = n0 - drop + 1;   // window after the push
    for (int i = tid; i < n - 1; i += ST_P1_THREADS) win[i] = st[8 + i + drop];
    const int pdrop = (p0 == ST_P) ? 1 : 0, np = p0 - pdrop + 1;
    for (int i = tid; i < np - 1; i += ST_P1_THREADS) pk[i] = (float)st[8 + ST_I + i + pdrop];
    if (tid == 0) { win[n - 1] = nv; pk[np - 1] = ntp; }
    __syncthreads();
    int nsort = 32;
    while (nsort < n) nsort <<= 1;
    int c = 0;
    double si = 0.0;
    for (int i = tid; i < nsort; i += ST_P1_THREADS) {
        const double v = (i < n) ? win[i] : 0.0;
        const bool g = i < n && v > a.gate;
        const float vf = (float)v;
        srt[i] = g ? vf : CUDART_INF_F;                       // non-gated entries sort to the end
        if (g) { ++c; si += (double)vf; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { c += __shfl_xor_sync(0xffffffffu, c, o); si += __shfl_xor_sync(0xffffffffu, si, o); }
    if (lane == 0) { red_i[warp] = c; red_d[warp] = si; }
    __syncthreads();
    for (int k = 2; k <= nsort; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < nsort; i += ST_P1_THREADS) {
                const int l = i ^ j;
                if (l > i) {
                    const float x = srt[i], y = srt[l];
                    if ((x > y) == ((i & k) == 0)) { srt[i] = y; srt[l] = x; }
                }
            }
            __syncthreads();
        }
    // new state: window and peak ring (every old value was copied to shared memory above)
    for (int i = tid; i < n; i += ST_P1_THREADS) st[8 + i] = win[i];
    for (int i = tid; i < np; i += ST_P1_THREADS) st[8 + ST_I + i] = (double)pk[i];
    if (tid == 0) {
        int ns = 0;
        double sum_i = 0.0;
        for (int w = 0; w < ST_P1_THREADS / 32; ++w) { ns += red_i[w]; sum_i += red_d[w]; }
        const int cm = n < ST_M ? n : ST_M, cs = n < ST_S ? n : ST_S;
        double sum_m = 0.0, sum_s = 0.0;
        for (int i = n - cm; i < n; ++i) sum_m += (double)(float)win[i];
        for (int i = n - cs; i < n; ++i) sum_s += (double)(float)win[i];
        float m = -CUDART_INF_F;
        for (int i = 0; i < np; ++i) m = fmaxf(m, pk[i]);
        double cur[5];
        cur[0] = sum_m * (1.0 / (double)cm);
        cur[1] = sum_s * (1.0 / (double)cs);
        cur[2] = ns > 0 ? sum_i * (1.0 / (double)ns) : -100.0;
        cur[3] = ns > 0 ? st_percentile_f(srt, ns, 0.95) - st_percentile_f(srt, ns, 0.10) : 0.0;
        cur[4] = (double)m;
        float* orow = a.out + (size_t)ch * 5;
        for (int i = 0; i < 5; ++i) { orow[i] = (float)cur[i]; st[2 + i] = cur[i]; }
        st[0] = (double)n; st[1] = (double)np; st[7] = 1.0;
    }
}

template <bool CARRIED>
inline size_t stats_smem_bytes() { return (size_t)stw_smem<CARRIED>(); }

}  // namespace o4
