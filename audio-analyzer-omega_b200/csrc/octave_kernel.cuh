// octave_kernel.cuh -- per-channel one-third-octave band levels (IEC 61260-1 base-10 bands, 6th-order digital
// Butterworth band-pass per band) every 100 ms, plus the running Leq and the maximum block level (omega4_octave_*).
// An extension outside reference parity: the reference has no calibrated band levels.
// Definitions: DESIGN.md section 4.8; float64 oracle: oracle/octave_np.py.
//
// Push (one launch): octave_kernel, one warp per channel row.
//   Lane b < n_bands runs band b's three biquads; lane n_bands runs no filter and sums x^2 (the overall level);
//   lanes above that idle.  The row's samples are staged through shared memory, OCT_CHUNK at a time: each lane
//   loads OCT_CHUNK / 32 floats with coalesced 128-byte warp loads (the next chunk's loads are issued before the
//   current chunk is filtered), converts them to double once, and then every lane reads each sample as a
//   shared-memory broadcast.  So a sample is read from HBM once for all bands and converted once per warp.
//   Each section's numerator is taken as [1, 0, -1] (one zero at z = 1 and one at z = -1) and the band's gain G
//   (the product of the three sections' b0) is applied to the energy, not in the recursion; a band's cascade is
//   H = G (1 - z^-2)^3 / prod(1 + a1 z^-1 + a2 z^-2) whichever way the six zeros were paired into sections.
//   Direct form II transposed, float64:  y = x + s1;  s1 = -a1 y + s2;  s2 = -a2 y - x   (1 DADD + 2 DFMA),
//   three sections and one DFMA for the energy: 10 float64 instructions per lane and sample.
//   The carried state per (row, column) is exact (6 filter values, the partial block's energy, the energy of
//   all completed blocks, the largest block energy), so tiles of any length continue bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

namespace o4 {

constexpr int OCT_MAX_BANDS = 31;
constexpr int OCT_COEF = 8;                      // per lane: -a1, -a2 of the three sections, 2 G^2 / sub, 2 G^2
constexpr int OCT_COL_DOUBLES = 9;               // per (row, column): s[6], partial energy, completed energy, max
#ifndef OMEGA4_OCT_WARPS
#define OMEGA4_OCT_WARPS 4                       // warps (rows) per CTA (1, 2 and 4 measured: DESIGN 4.8)
#endif
constexpr int OCT_WARPS = OMEGA4_OCT_WARPS;
constexpr int OCT_CHUNK = 256;                   // samples staged per warp at a time
constexpr int OCT_PER_LANE = OCT_CHUNK / 32;

// doubles of carried state per row: the sample count T, then OCT_COL_DOUBLES arrays of n_bands + 1 columns
__host__ __device__ inline int oct_state_doubles(int nb) { return 1 + OCT_COL_DOUBLES * (nb + 1); }

struct OctArgs {
    const float* x;            // [n_rows] rows of n samples, row r at x + r * ch_stride
    long long ch_stride;
    long long n;
    int n_rows, nb, sub;
    const double* coef;        // [32][OCT_COEF]
    double* state;             // [n_rows][oct_state_doubles(nb)]
    int fresh;
    float* levels;             // [n_rows][out_stride][nb + 1] or nullptr
    long long out_stride;
    float* leq;                // [n_rows][nb + 1] or nullptr
    float* lmax;
};

__device__ inline float oct_db(double e) { return (float)(10.0 * log10(e)); }   // -inf for e == 0

__global__ void __launch_bounds__(OCT_WARPS * 32) octave_kernel(OctArgs a) {
    __shared__ double xs[OCT_WARPS][OCT_CHUNK];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * OCT_WARPS + warp;
    if (row >= a.n_rows) return;                           // the whole warp leaves; only __syncwarp below
    const int ncol = a.nb + 1;
    const bool own = lane < ncol;
    const bool overall = lane == a.nb;
    const double* cf = a.coef + lane * OCT_COEF;
    const double c0 = cf[0], c1 = cf[1], c2 = cf[2], c3 = cf[3], c4 = cf[4], c5 = cf[5];
    const double sb = cf[6], se = cf[7];
    const double* st0 = a.state + row * oct_state_doubles(a.nb);
    const long long T = a.fresh ? 0 : (long long)st0[0];
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0, s5 = 0.0, acc = 0.0, etot = 0.0, emax = 0.0;
    if (!a.fresh && own) {
        const double* f = st0 + 1 + lane;
        s0 = f[0]; s1 = f[ncol]; s2 = f[2 * ncol]; s3 = f[3 * ncol]; s4 = f[4 * ncol]; s5 = f[5 * ncol];
        acc = f[6 * ncol]; etot = f[7 * ncol]; emax = f[8 * ncol];
    }
    long long left = a.sub - T % a.sub;                    // samples to the end of the current block
    long long col = 0;                                     // output column of the next completed block
    const float* xr = a.x + row * a.ch_stride;
    const long long n = a.n;
    float pre[OCT_PER_LANE];
#pragma unroll
    for (int k = 0; k < OCT_PER_LANE; ++k) {
        const long long idx = lane + 32 * k;
        pre[k] = idx < n ? __ldg(xr + idx) : 0.f;
    }
    for (long long c0i = 0; c0i < n; c0i += OCT_CHUNK) {
        __syncwarp();                                      // every lane is done with the previous chunk
#pragma unroll
        for (int k = 0; k < OCT_PER_LANE; ++k) xs[warp][lane + 32 * k] = (double)pre[k];
        __syncwarp();
        const long long nxt = c0i + OCT_CHUNK;
#pragma unroll
        for (int k = 0; k < OCT_PER_LANE; ++k) {
            const long long idx = nxt + lane + 32 * k;
            pre[k] = idx < n ? __ldg(xr + idx) : 0.f;
        }
        const int len = (int)(n - c0i < OCT_CHUNK ? n - c0i : OCT_CHUNK);
        int i = 0;
        while (i < len) {
            const int r = (int)(len - i < left ? len - i : left);
            const double* xp = &xs[warp][i];
#pragma unroll 4
            for (int k = 0; k < r; ++k) {
                const double xv = xp[k];
                const double y1 = xv + s0;
                s0 = fma(c0, y1, s1);
                s1 = fma(c1, y1, -xv);
                const double y2 = y1 + s2;
                s2 = fma(c2, y2, s3);
                s3 = fma(c3, y2, -y1);
                const double y3 = y2 + s4;
                s4 = fma(c4, y3, s5);
                s5 = fma(c5, y3, -y2);
                const double o = overall ? xv : y3;
                acc = fma(o, o, acc);
            }
            i += r;
            left -= r;
            if (left == 0) {                               // a block ends here
                if (own && a.levels && col < a.out_stride)
                    a.levels[(row * a.out_stride + col) * ncol + lane] = oct_db(sb * acc);
                etot += acc;
                emax = fmax(emax, acc);
                acc = 0.0;
                ++col;
                left = a.sub;
            }
        }
    }
    // the state pointer and T are re-derived here rather than kept live across the loop
    double* st = a.state + row * oct_state_doubles(a.nb);
    const long long Tn = (a.fresh ? 0 : (long long)st[0]) + n;
    __syncwarp();                                          // every lane has read T before lane 0 replaces it
    if (own) {
        double* f = st + 1 + lane;
        f[0] = s0; f[ncol] = s1; f[2 * ncol] = s2; f[3 * ncol] = s3; f[4 * ncol] = s4; f[5 * ncol] = s5;
        f[6 * ncol] = acc; f[7 * ncol] = etot; f[8 * ncol] = emax;
        if (a.leq) a.leq[row * ncol + lane] = oct_db(se * (etot + acc) / (double)Tn);
        if (a.lmax) a.lmax[row * ncol + lane] = oct_db(sb * emax);
    }
    if (lane == 0) st[0] = (double)Tn;
}

}  // namespace o4
