// loudness_kernel.cuh -- ITU-R BS.1770-4 program loudness and EBU Tech 3342 loudness range per stream
// (omega4_loudness_*).  An extension outside reference parity: the reference's ProfessionalMetering is
// not textbook BS.1770 (SURVEY.md section 0.2) and is served unchanged by the plan's meter kernels.
// Definitions: DESIGN.md section 4.7; float64 oracle: oracle/bs1770_np.py.
//
// Push (two launches):
//   loudness_chain_kernel     one thread per (channel row, run of LOUD_GROUP consecutive segments).  A
//       segment is the part of one 100 ms sub-block (sub = fs / 10 samples) that lies in the tile.  The thread
//       runs the K-weighting cascade (high-shelf, then high-pass; direct form II transposed, float64) from
//       max(tile start, start of its first segment - sub) to the end of its last segment and sums y^2
//       (float64) per segment.  Starting at the tile start it starts from the carried filter state, which is
//       exact; starting earlier than that it starts from zero one whole sub-block ahead, which leaves n r^n of
//       the true state (r = 0.99502 double pole of the high-pass at 48 kHz: 2e-7 at 48 and at 96 kHz, since
//       the warm-up is always 100 ms).  One warm-up per run of 8 segments: each input sample is read and
//       filtered 9/8 times, not twice.  Loads are staged through shared memory per warp: for each 32-sample
//       chunk the warp reads each of its 32 chains' 128 contiguous bytes with one coalesced instruction,
//       then every lane walks its own chain's 32 samples out of shared memory (stride 33, no conflicts).
//   loudness_finalize_kernel  one warp per stream: weighted sub-block energies z = sum_c G_c e_c (with the
//       carried partial sub-block), momentary / short-term loudness at every completed sub-block from z and
//       the carried 29 previous energies, then the carried state (sample count, energy history, filter
//       state, partial sub-block, sample peak).
// Summary (one launch): loudness_summary_kernel, one CTA per stream over the stored M / S series: the
// two-stage gating of the integrated loudness, the gates of the loudness range and its two percentiles as
// exact order statistics (4-pass 8-bit radix select over the order-preserving integer keys of the float values).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

namespace o4 {

constexpr int LOUD_MAX_CH = 32;
constexpr int LOUD_HIST = 29;                    // previous sub-block energies a short-term value needs
constexpr int LOUD_CH_DOUBLES = 6;               // per channel: shelf s1 s2, high-pass s1 s2, partial energy, peak
constexpr int LOUD_HDR = 1 + LOUD_HIST;          // per stream: sample count T, then z_{J-29} .. z_{J-1}
constexpr int LOUD_WARPS = 4;
constexpr int LOUD_GROUP = 8;                   // consecutive segments per thread of loudness_chain_kernel

__host__ __device__ inline int loud_state_doubles(int C) { return LOUD_HDR + LOUD_CH_DOUBLES * C; }

struct LoudArgs {
    const float* x;            // [n_streams * C] rows of n samples, row r at x + r * ch_stride
    long long ch_stride;
    long long n;
    int n_streams, C, sub;
    int nsegb;                 // segments per row the scratch is laid out for: n / sub + 2
    double sb0, sb1, sb2, sa1, sa2;    // high-shelf
    double hb0, hb1, hb2, ha1, ha2;    // high-pass
    double w[LOUD_MAX_CH];     // G_c
    double* state;             // [n_streams][loud_state_doubles(C)]
    int fresh;
    double* E;                 // [rows][nsegb] segment energies
    float* P;                  // [rows][nsegb] segment sample peaks
    double* FS;                // [rows][4] filter state at the tile end
    double* Z;                 // [n_streams][nsegb] weighted segment energies
    float* mom;                // [n_streams][out_stride] or nullptr
    float* st;
    long long out_stride;
    float* peak_db;            // [n_streams][C] or nullptr
};

__global__ void __launch_bounds__(LOUD_WARPS * 32) loudness_chain_kernel(LoudArgs a) {
    __shared__ float tile[LOUD_WARPS][32][33];
    __shared__ const float* cbase[LOUD_WARPS][32];
    __shared__ int clen[LOUD_WARPS][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long chain = ((long long)blockIdx.x * LOUD_WARPS + warp) * 32 + lane;
    const long long rows = (long long)a.n_streams * a.C;
    const long long ngroups = (a.nsegb + LOUD_GROUP - 1) / LOUD_GROUP;
    bool active = chain < rows * ngroups;
    long long row = 0, k = 0, nseg = 0, ws = 0;
    int L = 0, pre = 0, bnd = 0;
    const int SD = loud_state_doubles(a.C);
    double s1 = 0.0, s2 = 0.0, t1 = 0.0, t2 = 0.0;
    if (active) {
        row = chain / ngroups;
        k = (chain - row * ngroups) * LOUD_GROUP;          // first segment of this thread's run
        const long long s = row / a.C;
        const int c = (int)(row - s * a.C);
        const double* st = a.state + s * SD;
        const long long T = a.fresh ? 0 : (long long)st[0];
        const long long off = T % a.sub;
        nseg = (off + a.n + a.sub - 1) / a.sub;
        if (k >= nseg) {
            active = false;
        } else {
            const long long k1 = k + LOUD_GROUP < nseg ? k + LOUD_GROUP : nseg;
            const long long seg0 = k * a.sub - off > 0 ? k * a.sub - off : 0;
            const long long end = k1 * a.sub - off < a.n ? k1 * a.sub - off : a.n;
            const long long seg0_end = (k + 1) * a.sub - off < a.n ? (k + 1) * a.sub - off : a.n;
            ws = seg0 - a.sub > 0 ? seg0 - a.sub : 0;
            L = (int)(end - ws);
            pre = (int)(seg0 - ws);
            bnd = (int)(seg0_end - ws);                    // end of the current segment, relative to ws
            if (ws == 0 && !a.fresh) {
                const double* f = st + LOUD_HDR + LOUD_CH_DOUBLES * c;
                s1 = f[0]; s2 = f[1]; t1 = f[2]; t2 = f[3];
            }
        }
    }
    cbase[warp][lane] = active ? a.x + row * a.ch_stride + ws : nullptr;
    clen[warp][lane] = active ? L : 0;
    int maxL = L;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxL = max(maxL, __shfl_xor_sync(0xffffffffu, maxL, o));
    __syncwarp();
    double acc = 0.0;
    float pk = 0.f;
    for (int q = 0; q < maxL; q += 32) {
#pragma unroll 8
        for (int c = 0; c < 32; ++c) {
            const int idx = q + lane;
            tile[warp][c][lane] = idx < clen[warp][c] ? cbase[warp][c][idx] : 0.f;
        }
        __syncwarp();
        const int lim = L - q;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            if (i < lim) {
                const float v = tile[warp][lane][i];
                const double xv = (double)v;
                const double y1 = fma(a.sb0, xv, s1);
                s1 = fma(a.sb1, xv, fma(-a.sa1, y1, s2));
                s2 = fma(a.sb2, xv, -a.sa2 * y1);
                const double y2 = fma(a.hb0, y1, t1);
                t1 = fma(a.hb1, y1, fma(-a.ha1, y2, t2));
                t2 = fma(a.hb2, y1, -a.ha2 * y2);
                if (q + i >= pre) {
                    acc = fma(y2, y2, acc);
                    pk = fmaxf(pk, fabsf(v));
                }
                if (q + i + 1 == bnd) {                    // segment k ends here
                    a.E[row * a.nsegb + k] = acc;
                    a.P[row * a.nsegb + k] = pk;
                    acc = 0.0;
                    pk = 0.f;
                    ++k;
                    bnd = bnd + a.sub < L ? bnd + a.sub : L;
                }
            }
        }
        __syncwarp();
    }
    if (active && k == nseg) {                             // this run ended the tile: its state is carried
        double* f = a.FS + row * 4;
        f[0] = s1; f[1] = s2; f[2] = t1; f[3] = t2;
    }
}

__device__ inline float loud_lufs(double energy_per_sample) {
    return (float)(-0.691 + 10.0 * log10(energy_per_sample));
}

__global__ void __launch_bounds__(LOUD_WARPS * 32) loudness_finalize_kernel(LoudArgs a) {
    const int lane = threadIdx.x & 31;
    const long long s = (long long)blockIdx.x * LOUD_WARPS + (threadIdx.x >> 5);
    if (s >= a.n_streams) return;
    const int C = a.C, SD = loud_state_doubles(C);
    double* st = a.state + s * SD;
    const long long T = a.fresh ? 0 : (long long)st[0];
    const long long off = T % a.sub, J0 = T / a.sub;
    const long long nseg = (off + a.n + a.sub - 1) / a.sub;
    const long long ndone = (off + a.n) / a.sub;
    const long long rem = (off + a.n) % a.sub;
    double* Z = a.Z + s * a.nsegb;
    for (long long k = lane; k < nseg; k += 32) {
        double z = 0.0;
        for (int c = 0; c < C; ++c) {
            double e = a.E[(s * C + c) * a.nsegb + k];
            if (k == 0 && !a.fresh) e += st[LOUD_HDR + LOUD_CH_DOUBLES * c + 4];
            z = fma(a.w[c], e, z);
        }
        Z[k] = z;
    }
    __syncwarp();
    const double inv4 = 1.0 / (4.0 * a.sub), inv30 = 1.0 / (30.0 * a.sub);
    for (long long jl = lane; jl < ndone; jl += 32) {
        const long long j = J0 + jl;
        double sm = 0.0, ss = 0.0;
        for (long long i = j - LOUD_HIST; i <= j; ++i) {
            if (i < 0) continue;
            const double z = i >= J0 ? Z[i - J0] : st[1 + LOUD_HIST - (J0 - i)];
            ss += z;
            if (i >= j - 3) sm += z;
        }
        const float M = j >= 3 ? loud_lufs(sm * inv4) : CUDART_NAN_F;
        const float S = j >= LOUD_HIST ? loud_lufs(ss * inv30) : CUDART_NAN_F;
        if (a.mom && jl < a.out_stride) a.mom[s * a.out_stride + jl] = M;
        if (a.st && jl < a.out_stride) a.st[s * a.out_stride + jl] = S;
    }
    // carried state: every read of the old state above happens before any write below
    double h = 0.0;
    if (lane < LOUD_HIST) {
        const long long idx = ndone + lane;
        h = idx < LOUD_HIST ? (a.fresh ? 0.0 : st[1 + idx]) : Z[idx - LOUD_HIST];
    }
    // C <= LOUD_MAX_CH = 32: lane c owns channel c
    double part = 0.0;
    float pk = 0.f;
    if (lane < C) {
        const double* f = st + LOUD_HDR + LOUD_CH_DOUBLES * lane;
        const long long r = s * C + lane;
        if (rem != 0) part = (nseg == 1 && !a.fresh ? f[4] : 0.0) + a.E[r * a.nsegb + nseg - 1];
        pk = a.fresh ? 0.f : (float)f[5];
        for (long long k = 0; k < nseg; ++k) pk = fmaxf(pk, a.P[r * a.nsegb + k]);
    }
    __syncwarp();
    if (lane < LOUD_HIST) st[1 + lane] = h;
    if (lane < C) {
        double* f = st + LOUD_HDR + LOUD_CH_DOUBLES * lane;
        const double* fs = a.FS + (s * C + lane) * 4;
        f[0] = fs[0]; f[1] = fs[1]; f[2] = fs[2]; f[3] = fs[3];
        f[4] = part; f[5] = pk;
        if (a.peak_db) a.peak_db[s * C + lane] = pk > 0.f ? (float)(20.0 * log10((double)pk)) : -CUDART_INF_F;
    }
    if (lane == 0) st[0] = (double)(T + a.n);
}

// ---- summary -----------------------------------------------------------------------------------------
constexpr int LOUD_SUM_THREADS = 256;

__device__ inline unsigned loud_key(float v) {
    const unsigned u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ inline float loud_unkey(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

template <typename T, typename Op>
__device__ T loud_block_reduce(T v, Op op, T* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();                          // sh may still be read by the previous reduction
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    T r = sh[0];
    for (int i = 1; i < LOUD_SUM_THREADS / 32; ++i) r = op(r, sh[i]);
    return r;
}

struct LoudGate {
    double mean_energy;   // energy mean of the values above the gate(s), 0 when none
    int count;
};

// energy mean / count of the values v > -70 and v > rel (NaN and -inf never pass)
__device__ LoudGate loud_gate(const float* v, int n, double rel, double* shd, int* shi) {
    double e = 0.0;
    int cnt = 0;
    for (int j = threadIdx.x; j < n; j += LOUD_SUM_THREADS) {
        const float x = v[j];
        if (x > -70.f && (double)x > rel) { e += exp10(((double)x + 0.691) / 10.0); ++cnt; }
    }
    e = loud_block_reduce(e, [](double p, double q) { return p + q; }, shd);
    cnt = loud_block_reduce(cnt, [](int p, int q) { return p + q; }, shi);
    return {cnt ? e / cnt : 0.0, cnt};
}

__device__ inline double loud_lufs_d(double e) { return -0.691 + 10.0 * log10(e); }

// k-th smallest (0-based) of the values passing (v > -70 && v > rel); k < their count
__device__ float loud_select(const float* v, int n, double rel, unsigned k, unsigned* hist, unsigned* sel) {
    unsigned prefix = 0u, mask = 0u;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = threadIdx.x; i < 256; i += LOUD_SUM_THREADS) hist[i] = 0u;
        __syncthreads();
        for (int j = threadIdx.x; j < n; j += LOUD_SUM_THREADS) {
            const float x = v[j];
            if (x > -70.f && (double)x > rel) {
                const unsigned key = loud_key(x);
                if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned cum = 0u;
            int b = 0;
            for (; b < 255; ++b) {
                if (cum + hist[b] > k) break;
                cum += hist[b];
            }
            sel[0] = prefix | ((unsigned)b << shift);
            sel[1] = k - cum;
        }
        __syncthreads();
        prefix = sel[0];
        k = sel[1];
        mask |= 255u << shift;
        __syncthreads();
    }
    return loud_unkey(prefix);
}

// momentary / short_term [n_streams][stride] series of n_steps values -> out [n_streams][4] = I, LRA, max M, max S
__global__ void __launch_bounds__(LOUD_SUM_THREADS) loudness_summary_kernel(const float* mom, const float* sht,
                                                                            long long stride, int n_steps, float* out) {
    __shared__ double shd[LOUD_SUM_THREADS / 32];
    __shared__ int shi[LOUD_SUM_THREADS / 32];
    __shared__ float shf[LOUD_SUM_THREADS / 32];
    __shared__ unsigned hist[256], sel[2];
    const long long s = blockIdx.x;
    const float* m = mom + s * stride;
    const float* sh = sht + s * stride;
    float mx_m = -CUDART_INF_F, mx_s = -CUDART_INF_F;
    int def_m = 0, def_s = 0;
    for (int j = threadIdx.x; j < n_steps; j += LOUD_SUM_THREADS) {
        if (!isnan(m[j])) { mx_m = fmaxf(mx_m, m[j]); ++def_m; }
        if (!isnan(sh[j])) { mx_s = fmaxf(mx_s, sh[j]); ++def_s; }
    }
    auto fmax_op = [](float p, float q) { return fmaxf(p, q); };
    auto add_i = [](int p, int q) { return p + q; };
    mx_m = loud_block_reduce(mx_m, fmax_op, shf);
    def_m = loud_block_reduce(def_m, add_i, shi);
    mx_s = loud_block_reduce(mx_s, fmax_op, shf);
    def_s = loud_block_reduce(def_s, add_i, shi);

    // integrated loudness: absolute gate, then 10 LU below the energy mean of the survivors
    LoudGate g = loud_gate(m, n_steps, -CUDART_INF, shd, shi);
    float I = -CUDART_INF_F;
    if (g.count) {
        const LoudGate g2 = loud_gate(m, n_steps, loud_lufs_d(g.mean_energy) - 10.0, shd, shi);
        if (g2.count) I = (float)loud_lufs_d(g2.mean_energy);
    }
    // loudness range: absolute gate, then 20 LU below the energy mean; percentiles 10 and 95 (rounded ranks)
    float lra = 0.f;
    g = loud_gate(sh, n_steps, -CUDART_INF, shd, shi);
    if (g.count) {
        const double rel = loud_lufs_d(g.mean_energy) - 20.0;
        const LoudGate g2 = loud_gate(sh, n_steps, rel, shd, shi);
        if (g2.count) {
            const double nm1 = (double)(g2.count - 1);
            const unsigned k_lo = (unsigned)floor(0.10 * nm1 + 0.5), k_hi = (unsigned)floor(0.95 * nm1 + 0.5);
            const float lo = loud_select(sh, n_steps, rel, k_lo, hist, sel);
            const float hi = loud_select(sh, n_steps, rel, k_hi, hist, sel);
            lra = (float)((double)hi - (double)lo);
        }
    }
    if (threadIdx.x == 0) {
        out[s * 4 + 0] = I;
        out[s * 4 + 1] = lra;
        out[s * 4 + 2] = def_m ? mx_m : CUDART_NAN_F;
        out[s * 4 + 3] = def_s ? mx_s : CUDART_NAN_F;
    }
}

}  // namespace o4
