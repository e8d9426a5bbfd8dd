// idelucs_b200 — per-sample silhouette coefficients (sklearn.metrics.silhouette_samples, metric "euclidean") of a
// float32 [n, D] matrix under a labelling; DESIGN.md §4, K10.
//
// Exactness: d(i, j) is the distance of the HDBSCAN kernels (pairwise.cuh: fp64, sum in order over t, no FMA, IEEE
// sqrt).  S_c(i), the sum of d(i, j) over the points j of cluster c, is a left fold in increasing j, self included:
// the order of sklearn's np.bincount.  The silhouette then follows sklearn's formula with IEEE divisions.
//
// The host groups the points by label (a stable counting sort) and the kernel walks every row's n columns in that
// order: a CTA owns BI = 64 rows in the original order, sq_tile gathers the columns through the order array, the
// distances of a tile go to shared memory, and one thread per row folds them.  At every cluster boundary that thread
// finalises the cluster as the row's own (intra) or as a candidate for the nearest other cluster (inter), so its state
// is O(1) whatever the number of clusters and nothing of size n x n or n x n_labels is stored.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include <vector>

#include "../../include/idelucs_b200.h"
#include "common.h"
#include "pairwise.cuh"

namespace idl {
namespace {

constexpr long long SIL_MAX_N = 0x7fffffffLL;   // column positions and cluster offsets are int32

struct SilSmem {
    Panels p;
    double d[BI][BJ + 1];   // distances of the current tile, row-major
};

// out[i] = silhouette of row i for the rows of [row_begin, row_end) (CTA b owns row_begin + 64 b ..); order: int32[n], the
// points in label-sorted order (stable); off: int32[n_labels + 1], cluster c holds the positions off[c] .. off[c + 1] - 1 of `order`
__global__ void __launch_bounds__(NT) silhouette_kernel(const float* __restrict__ x, const int* __restrict__ labels, long long n, int D,
                                                        long long row_begin, long long row_end, const int* __restrict__ order,
                                                        const int* __restrict__ off, double* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem[];
    SilSmem& s = *reinterpret_cast<SilSmem*>(smem);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const long long row0 = row_begin + (long long)blockIdx.x * BI;
    // the fold state of row row0 + threadIdx.x (threads < BI)
    const long long i = row0 + threadIdx.x;
    const bool folds = threadIdx.x < BI && i < row_end;
    const int own = folds ? labels[i] : -1;
    int c = 0;                     // the cluster of the next column position
    long long end = folds ? off[1] : 0;   // its end position
    double S = 0.0, intra = 0.0, inter = INFINITY;
    long long n_own = 0;
    auto finalise = [&]() {        // cluster c is complete: S = S_c(i)
        const long long nc = end - off[c];
        if (c == own) {
            intra = S;
            n_own = nc;
        } else if (nc > 0) {
            const double v = S / (double)nc;
            if (v < inter) inter = v;
        }
        S = 0.0;
        ++c;
    };

    double acc[4][4];
    for (long long col0 = 0; col0 < n; col0 += BJ) {
        sq_tile(x, n, D, row0, col0, s.p, acc, Gather{order});
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) s.d[ty + 16 * r][tx + 16 * cc] = __dsqrt_rn(acc[r][cc]);
        __syncthreads();
        if (folds) {
            const int nq = (int)min((long long)BJ, n - col0);
            int q = 0;
            while (q < nq) {
                if (col0 + q >= end) {   // a cluster boundary (empty clusters pass here too)
                    finalise();
                    end = off[c + 1];
                    continue;
                }
                const int lim = (int)min((long long)nq, end - col0);
                for (; q < lim; ++q) S = __dadd_rn(S, s.d[threadIdx.x][q]);
            }
        }
        // the next sq_tile starts with a barrier, so s.d is not overwritten before every row has read it
    }
    if (!folds) return;
    finalise();   // the last non-empty cluster; any clusters after it are empty
    double v = 0.0;
    if (n_own > 1) {
        intra = intra / (double)(n_own - 1);
        v = (inter - intra) / fmax(intra, inter);
        if (isnan(v)) v = 0.0;   // intra = inter = 0 (or no other cluster): sklearn's nan_to_num
    }
    out[i] = v;
}

constexpr size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
constexpr size_t SIL_SMEM = sizeof(SilSmem);

// silhouette of the rows of [row_begin, row_end) (arguments already checked except the label values)
int silhouette_rows(const char* who, const float* d_x, const int32_t* d_labels, int64_t n, int D, int64_t n_labels, int64_t row_begin,
                    int64_t row_end, double* d_out, void* d_ws, cudaStream_t st) {
    // group the points by label on the host: a stable counting sort
    std::vector<int32_t> lab(n);
    IDL_CUDA_CHECK(cudaMemcpyAsync(lab.data(), d_labels, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    IDL_CUDA_CHECK(cudaStreamSynchronize(st));
    std::vector<int32_t> off(n_labels + 1, 0), order(n);
    for (int64_t i = 0; i < n; ++i) {
        if (lab[i] < 0 || lab[i] >= n_labels) {
            char what[96];
            snprintf(what, sizeof(what), "%s: label %d outside 0..%lld", who, (int)lab[i], (long long)(n_labels - 1));
            return set_error(IDL_EINVAL, "%s at position %lld", what, (long long)i);
        }
        ++off[lab[i] + 1];
    }
    if (row_end == row_begin) return IDL_OK;
    for (int64_t c = 0; c < n_labels; ++c) off[c + 1] += off[c];
    {
        std::vector<int32_t> fill(off.begin(), off.end() - 1);
        for (int64_t i = 0; i < n; ++i) order[fill[lab[i]]++] = (int32_t)i;
    }
    char* ws = reinterpret_cast<char*>(d_ws);
    int* d_order = reinterpret_cast<int*>(ws);
    int* d_off = reinterpret_cast<int*>(ws + align256((size_t)n * sizeof(int)));
    // pageable sources: each copy returns once its source has been staged, so the host vectors may die on return
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_order, order.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_off, off.data(), (n_labels + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));

    IDL_CUDA_CHECK(cudaFuncSetAttribute(silhouette_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SIL_SMEM));
    silhouette_kernel<<<(unsigned)((row_end - row_begin + BI - 1) / BI), NT, SIL_SMEM, st>>>(d_x, d_labels, n, D, row_begin, row_end, d_order,
                                                                                           d_off, d_out);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int check_args(const char* who, const float* d_x, const int32_t* d_labels, int64_t n, int D, int64_t n_labels, const double* d_out,
               const void* d_ws) {
    if (!d_x || !d_labels || !d_out || !d_ws) return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (n < 1 || n > SIL_MAX_N) return set_error(IDL_EINVAL, "%s: n must be in 1..2147483647 (got %lld)", who, (long long)n);
    if (D < 1) return set_error(IDL_EINVAL, "%s: D must be >= 1 (got %lld)", who, (long long)D);
    if (n_labels < 1 || n_labels > n) return set_error(IDL_EINVAL, "%s: n_labels must be in 1..n (got %lld)", who, (long long)n_labels);
    return IDL_OK;
}

int check_ws(const char* who, int64_t n, int64_t n_labels, size_t ws_bytes) {
    const size_t need = idl_silhouette_workspace_bytes(n, n_labels);
    if (ws_bytes < need) return set_error(IDL_EINVAL, "%s: workspace too small (need %lld bytes)", who, (long long)need);
    return IDL_OK;
}

}  // namespace
}  // namespace idl

using namespace idl;

extern "C" size_t idl_silhouette_workspace_bytes(int64_t n, int64_t n_labels) {
    if (n < 1 || n > SIL_MAX_N || n_labels < 1 || n_labels > n) return 0;
    return align256((size_t)n * sizeof(int)) + align256((size_t)(n_labels + 1) * sizeof(int));
}

extern "C" int idl_silhouette_samples(const float* d_x, const int32_t* d_labels, int64_t n, int D, int64_t n_labels, double* d_out, void* d_ws,
                                      size_t ws_bytes, void* stream) {
    static const char* who = "idl_silhouette_samples";
    if (int rc = check_args(who, d_x, d_labels, n, D, n_labels, d_out, d_ws)) return rc;
    if (int rc = check_ws(who, n, n_labels, ws_bytes)) return rc;
    return silhouette_rows(who, d_x, d_labels, n, D, n_labels, 0, n, d_out, d_ws, (cudaStream_t)stream);
}

extern "C" int idl_silhouette_samples_rows(const float* d_x, const int32_t* d_labels, int64_t n, int D, int64_t n_labels, int64_t row_begin,
                                           int64_t row_end, double* d_out, void* d_ws, size_t ws_bytes, void* stream) {
    static const char* who = "idl_silhouette_samples_rows";
    if (int rc = check_args(who, d_x, d_labels, n, D, n_labels, d_out, d_ws)) return rc;
    if (int rc = check_rows(who, n, row_begin, row_end)) return rc;
    if (int rc = check_ws(who, n, n_labels, ws_bytes)) return rc;
    return silhouette_rows(who, d_x, d_labels, n, D, n_labels, row_begin, row_end, d_out, d_ws, (cudaStream_t)stream);
}
