// idelucs_b200 — the exact fp64 distance tile shared by the all-pairs kernels (hdbscan.cu, metrics.cu).
//
// A CTA of NT = 256 threads owns BI = 64 rows and walks the columns in BJ = 64-column tiles; the two 64 x DT fp64
// panels sit in shared memory and every thread accumulates a 4 x 4 micro-tile of squared distances.  The sum runs over
// t = 0..D-1 in order with every operation rounded on its own (__dsub_rn / __dmul_rn / __dadd_rn, never contracted
// into an FMA): the arithmetic of sklearn's EuclideanDistance once an IEEE sqrt is applied.
#pragma once
#include <cuda_runtime.h>

namespace idl {
namespace {

constexpr int BI = 64, BJ = 64, DT = 32, NT = 256;

struct Panels {
    double a[DT][BI + 1];   // +1: the transposed stores of the loader hit distinct banks
    double b[DT][BJ + 1];
};

// column position -> row of x: the identity, or a gather through an index array
struct SameOrder {
    __device__ __forceinline__ long long operator()(long long j) const { return j; }
};
struct Gather {
    const int* __restrict__ idx;
    __device__ __forceinline__ long long operator()(long long j) const { return idx[j]; }
};

// acc[r][c] = squared distance of rows row0 + ty + 16 r and columns col0 + tx + 16 c (0 outside [0, n)); column
// position j is row col(j) of x
template <typename Col = SameOrder>
__device__ __forceinline__ void sq_tile(const float* __restrict__ x, long long n, int D, long long row0, long long col0, Panels& s,
                                        double acc[4][4], Col col = Col()) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
    for (int t0 = 0; t0 < D; t0 += DT) {
        __syncthreads();
        for (int e = threadIdx.x; e < DT * BI; e += NT) {
            const int rr = e / DT, t = e % DT;
            const long long gi = row0 + rr, gj = col0 + rr;
            const bool tin = t0 + t < D;
            s.a[t][rr] = (tin && gi < n) ? (double)x[gi * D + t0 + t] : 0.0;
            s.b[t][rr] = (tin && gj < n) ? (double)x[col(gj) * D + t0 + t] : 0.0;
        }
        __syncthreads();
        const int tn = min(DT, D - t0);
        for (int t = 0; t < tn; ++t) {
            double av[4], bv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) av[r] = s.a[t][ty + 16 * r];
#pragma unroll
            for (int c = 0; c < 4; ++c) bv[c] = s.b[t][tx + 16 * c];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const double df = __dsub_rn(av[r], bv[c]);
                    acc[r][c] = __dadd_rn(acc[r][c], __dmul_rn(df, df));
                }
        }
    }
}

}  // namespace
}  // namespace idl
