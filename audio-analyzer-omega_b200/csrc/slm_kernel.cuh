// slm_kernel.cuh -- per-channel IEC 61672-1 sound level meter (omega4_slm_*): A, C and Z frequency weighting, Fast
// and Slow exponential time weighting, every 100 ms Leq, LFmax, LSmax, LF, LS and Lpeak per weighting, running
// totals, and percentile levels L_N of any series column.  An extension outside reference parity: the reference's
// A / C / Z meters are frame-wise zero-phase filters without time weighting and stay as they are.
// Definitions: DESIGN.md section 4.9; float64 oracle: oracle/slm_np.py.
//
// Push (one launch): slm_kernel, one CTA per 32 channel rows, three warps: warp 0 runs A, warp 1 C, warp 2 Z,
//   lane l of each warp owns row l of the CTA.  Every warp runs one uniform program.  The 32 rows are staged
//   through shared memory SLM_CHUNK samples at a time (double-buffered, one __syncthreads per chunk): each warp
//   loads rows warp, warp + 3, ... with one coalesced 128-byte instruction per row, converts to double once, and
//   lane l then walks row l out of the [32][33] tile (stride 33 doubles: no bank conflicts).  So a sample is read
//   from HBM once per CTA for all three weightings.
//   Each weighting section runs as numerator [1, m, 1], m = +2 or -2 (two zeros at z = -1 or at z = 1), direct form
//   II transposed in float64:  y = x + s1;  s1 = -a1 y + (m x + s2);  s2 = -a2 y + x   (1 DADD + 3 DFMA).  The
//   cascade's gain G (the product of the sections' b0) is applied at output time: G^2 to energies, which carries
//   the peak as well (max y^2).  Per sample after the sections: e = y^2, the block energy, v = fma(a, v - e, e) for
//   F and S, and three linear-domain maxima (v_F, v_S, e).  Logs are taken only at block ends and at the push end.
//   The carried state per row (the sample count T, per weighting the filter values, v_F, v_S, the partial block's
//   energy and maxima, and the running totals) is exact, so any cut of a stream into pushes is bit-identical.
// Percentiles (one launch): slm_percentile_kernel, one CTA per row, for each requested N an exact 4-pass 8-bit radix
//   select over the order-preserving integer keys (loud_key / loud_unkey of loudness_kernel.cuh) of the column.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

#include "loudness_kernel.cuh"

namespace o4 {

constexpr int SLM_NW = 3;                        // weightings, in the order A, C, Z
constexpr int SLM_NQ = 6;                        // per block and weighting: Leq, LFmax, LSmax, LF, LS, Lpeak
constexpr int SLM_NCOL = SLM_NW * SLM_NQ;        // series columns per block
constexpr int SLM_NTOT = 4;                      // totals per weighting: Leq, LFmax, LSmax, Lpeak
constexpr int SLM_MAX_SEC = 3;                   // sections of A; C has 2, Z none
constexpr int SLM_ROWS = 32;                     // rows per CTA
constexpr int SLM_CHUNK = 32;                    // samples per row staged at a time
constexpr int SLM_LOADS = (SLM_ROWS + SLM_NW - 1) / SLM_NW;   // rows each warp loads per chunk
// per weighting after its 2 * n_sections filter values: v_F, v_S, the partial block's energy, its max v_F, max v_S
// and max e, then the total energy of the completed blocks and their max v_F, max v_S and max e
constexpr int SLM_ACC = 10;
constexpr int SLM_STATE_DOUBLES = 1 + 2 * (3 + 2 + 0) + SLM_NW * SLM_ACC;      // 41
constexpr int SLM_PCT_THREADS = 256;
constexpr int SLM_MAX_PCT = 64;

__host__ __device__ constexpr int slm_sections(int w) { return w == 0 ? 3 : w == 1 ? 2 : 0; }
__host__ __device__ constexpr int slm_state_offset(int w) {   // first double of weighting w's state in a row
    return w == 0 ? 1 : w == 1 ? 1 + 6 + SLM_ACC : 1 + 6 + 4 + 2 * SLM_ACC;
}

struct SlmCoef {
    double m[SLM_MAX_SEC];     // numerator middle tap b1 / b0: +2 or -2
    double na1[SLM_MAX_SEC];   // -a1
    double na2[SLM_MAX_SEC];   // -a2
    double g2;                 // G^2
    double g2_sub;             // G^2 / sub
};

struct SlmArgs {
    const float* x;            // [n_rows] rows of n samples, row r at x + r * ch_stride
    long long ch_stride;
    long long n;
    int n_rows, sub;
    double aF, aS;             // exp(-1 / (tau fs)) for tau = 0.125 s and 1 s
    SlmCoef w[SLM_NW];
    double* state;             // [n_rows][SLM_STATE_DOUBLES]
    int fresh;
    float* levels;             // [n_rows][out_stride][SLM_NW][SLM_NQ] or nullptr
    long long out_stride;
    float* totals;             // [n_rows][SLM_NW][SLM_NTOT] or nullptr
};

struct SlmAcc {
    double s[2 * SLM_MAX_SEC];
    double vF, vS, e, mF, mS, mP;    // e: the partial block's energy
};

__device__ inline float slm_db(double e) { return (float)(10.0 * log10(e)); }   // -inf for e == 0

// r samples of weighting W from xp[0 .. r)
template <int W>
__device__ __forceinline__ void slm_span(const SlmArgs& a, const double* xp, int r, SlmAcc& q) {
    constexpr int NS = slm_sections(W);
#pragma unroll 4
    for (int k = 0; k < r; ++k) {
        double y = xp[k];
#pragma unroll
        for (int j = 0; j < NS; ++j) {
            const double u = y;
            y = u + q.s[2 * j];
            q.s[2 * j] = fma(a.w[W].na1[j], y, fma(a.w[W].m[j], u, q.s[2 * j + 1]));
            q.s[2 * j + 1] = fma(a.w[W].na2[j], y, u);
        }
        const double e = y * y;
        q.e += e;
        q.vF = fma(a.aF, q.vF - e, e);
        q.vS = fma(a.aS, q.vS - e, e);
        q.mF = fmax(q.mF, q.vF);
        q.mS = fmax(q.mS, q.vS);
        q.mP = fmax(q.mP, e);
    }
}

__global__ void __launch_bounds__(SLM_NW * 32, 1) slm_kernel(SlmArgs a) {
    __shared__ double xs[2][SLM_ROWS][SLM_CHUNK + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long r0 = (long long)blockIdx.x * SLM_ROWS;
    const long long row = r0 + lane;
    const bool valid = row < a.n_rows;
    const int ns = slm_sections(warp), off = slm_state_offset(warp);
    const double g2 = a.w[warp].g2, g2_sub = a.w[warp].g2_sub;
    const long long T = a.fresh ? 0 : (long long)a.state[r0 * SLM_STATE_DOUBLES];
    SlmAcc q = {};
    double etot = 0.0, tF = 0.0, tS = 0.0, tP = 0.0;
    if (valid && !a.fresh) {
        const double* f = a.state + row * SLM_STATE_DOUBLES + off;
#pragma unroll
        for (int j = 0; j < 2 * SLM_MAX_SEC; ++j)
            if (j < 2 * ns) q.s[j] = f[j];
        f += 2 * ns;
        q.vF = f[0]; q.vS = f[1]; q.e = f[2]; q.mF = f[3]; q.mS = f[4]; q.mP = f[5];
        etot = f[6]; tF = f[7]; tS = f[8]; tP = f[9];
    }
    const long long n = a.n;
    float pre[SLM_LOADS];
    auto load = [&](long long c0) {
#pragma unroll
        for (int i = 0; i < SLM_LOADS; ++i) {
            const int c = warp + SLM_NW * i;
            const long long idx = c0 + lane;
            pre[i] = (c < SLM_ROWS && r0 + c < a.n_rows && idx < n) ? __ldg(a.x + (r0 + c) * a.ch_stride + idx) : 0.f;
        }
    };
    auto stage = [&](int b) {
#pragma unroll
        for (int i = 0; i < SLM_LOADS; ++i) {
            const int c = warp + SLM_NW * i;
            if (c < SLM_ROWS) xs[b][c][lane] = (double)pre[i];
        }
    };
    load(0);
    stage(0);
    __syncthreads();
    load(SLM_CHUNK);
    long long left = a.sub - T % a.sub;                    // samples to the end of the current block
    long long col = 0;                                     // output column of the next completed block
    int b = 0;
    for (long long c0 = 0; c0 < n; c0 += SLM_CHUNK, b ^= 1) {
        stage(b ^ 1);                                      // chunk c0 + SLM_CHUNK: its buffer was last read before
        load(c0 + 2 * SLM_CHUNK);                          // the previous __syncthreads
        const int len = (int)(n - c0 < SLM_CHUNK ? n - c0 : SLM_CHUNK);
        int i = 0;
        while (i < len) {
            const int r = (int)(len - i < left ? len - i : left);
            const double* xp = &xs[b][lane][i];
            if (warp == 0) slm_span<0>(a, xp, r, q);
            else if (warp == 1) slm_span<1>(a, xp, r, q);
            else slm_span<2>(a, xp, r, q);
            i += r;
            left -= r;
            if (left == 0) {                               // a block ends here
                if (valid && a.levels && col < a.out_stride) {
                    float* o = a.levels + ((row * a.out_stride + col) * SLM_NW + warp) * SLM_NQ;
                    o[0] = slm_db(g2_sub * q.e);
                    o[1] = slm_db(g2 * q.mF);
                    o[2] = slm_db(g2 * q.mS);
                    o[3] = slm_db(g2 * q.vF);
                    o[4] = slm_db(g2 * q.vS);
                    o[5] = slm_db(g2 * q.mP);
                }
                etot += q.e;
                tF = fmax(tF, q.mF);
                tS = fmax(tS, q.mS);
                tP = fmax(tP, q.mP);
                q.e = q.mF = q.mS = q.mP = 0.0;
                ++col;
                left = a.sub;
            }
        }
        __syncthreads();                                   // every warp is done with buffer b before it is restaged
    }
    // the CTA's every thread read T above, before the __syncthreads of the loop (n > 0)
    if (valid) {
        double* f = a.state + row * SLM_STATE_DOUBLES + off;
#pragma unroll
        for (int j = 0; j < 2 * SLM_MAX_SEC; ++j)
            if (j < 2 * ns) f[j] = q.s[j];
        f += 2 * ns;
        f[0] = q.vF; f[1] = q.vS; f[2] = q.e; f[3] = q.mF; f[4] = q.mS; f[5] = q.mP;
        f[6] = etot; f[7] = tF; f[8] = tS; f[9] = tP;
        const long long Tn = T + n;
        if (a.totals) {
            float* o = a.totals + (row * SLM_NW + warp) * SLM_NTOT;
            o[0] = slm_db(g2 * (etot + q.e) / (double)Tn);
            o[1] = slm_db(g2 * fmax(tF, q.mF));
            o[2] = slm_db(g2 * fmax(tS, q.mS));
            o[3] = slm_db(g2 * fmax(tP, q.mP));
        }
        if (warp == 0) a.state[row * SLM_STATE_DOUBLES] = (double)Tn;
    }
}

// ---- percentiles -------------------------------------------------------------------------------------
struct SlmPctArgs {
    const float* levels;       // [n_rows][stride][SLM_NCOL]
    long long stride;
    int n_steps, column, n_pct;
    unsigned rank[SLM_MAX_PCT];   // 0-based ascending rank of each requested N among the n_steps values
    float* out;                // [n_rows][n_pct]
};

__global__ void __launch_bounds__(SLM_PCT_THREADS) slm_percentile_kernel(SlmPctArgs a) {
    __shared__ unsigned hist[256], sel[2];
    const long long r = blockIdx.x;
    const float* v = a.levels + r * a.stride * SLM_NCOL + a.column;
    for (int p = 0; p < a.n_pct; ++p) {
        if (a.n_steps == 0) {
            if (threadIdx.x == 0) a.out[r * a.n_pct + p] = CUDART_NAN_F;
            continue;
        }
        unsigned k = a.rank[p], prefix = 0u, mask = 0u;
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int i = threadIdx.x; i < 256; i += SLM_PCT_THREADS) hist[i] = 0u;
            __syncthreads();
            for (int j = threadIdx.x; j < a.n_steps; j += SLM_PCT_THREADS) {
                const unsigned key = loud_key(v[(long long)j * SLM_NCOL]);
                if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
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
        if (threadIdx.x == 0) a.out[r * a.n_pct + p] = loud_unkey(prefix);
    }
}

}  // namespace o4
