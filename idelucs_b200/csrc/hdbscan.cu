// idelucs_b200 — the all-pairs part of HDBSCAN (sklearn.cluster.HDBSCAN, metric "euclidean", alpha 1) over a float32
// [n, D] matrix: exact core distances (k-th smallest distance per row) and the minimum spanning tree of the implicit
// mutual-reachability graph w(i, j) = max(core[i], core[j], d(i, j)).  The condensed tree and cluster selection stay
// on the host (sklearn); DESIGN.md §4.8.
//
// Exactness: d(i, j) = sqrt(sum_t (x_i[t] - x_j[t])^2) with the float32 inputs widened to fp64, the sum taken in
// order t = 0..D-1 and every operation rounded on its own (__dsub_rn / __dmul_rn / __dadd_rn, never contracted into
// an FMA), then an IEEE sqrt.  That is the arithmetic of sklearn's EuclideanDistance, so core distances and MST
// weights compare with sklearn's by ==.
//
// Both passes share one tile loop (sq_tile, pairwise.cuh): a CTA owns BI = 64 rows and walks all n columns in BJ = 64-column
// tiles; the two 64 x DT fp64 panels sit in shared memory and every thread accumulates a 4 x 4 micro-tile of squared distances.
// Nothing of size n x n is ever stored: the core distances are a radix select over the fp64 bit patterns of the
// squared distances (non-negative doubles order like their bits, and sqrt is monotone), recomputing the distances on
// every pass; the MST is Borůvka, one all-pairs pass per round.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <numeric>
#include <vector>

#include "../../include/idelucs_b200.h"
#include "common.h"
#include "pairwise.cuh"

namespace idl {
namespace {

constexpr int BINS = 256;       // 8-bit radix digits: at most 8 passes over the 64-bit keys
constexpr int LIST_MAX = 128;   // a row whose candidate bucket holds <= this many keys collects them and finishes in one pass
constexpr int MODE_HIST = 0, MODE_LIST = 1, MODE_DONE = 2;
constexpr unsigned long long NONE = ~0ull;

// radix-select state of one row: the k-th smallest key has the top `nbits` bits of `prefix`; it is the `rank`-th
// smallest (1-based) of the `count` keys that share that prefix
struct RowSel {
    unsigned long long prefix;
    long long rank, count;
    int nbits, mode;
};

__global__ void core_init_kernel(RowSel* __restrict__ sel, long long n, long long k) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) sel[i] = RowSel{0ull, k, n, 0, n <= LIST_MAX ? MODE_LIST : MODE_HIST};
}

// one radix-select pass: every unfinished row either histograms the next 8-bit digit of the keys that match its prefix
// (MODE_HIST) or collects those keys and picks the rank-th (MODE_LIST).  CTAs whose rows are all done return at once.
__global__ void __launch_bounds__(NT) core_pass_kernel(const float* __restrict__ x, long long n, int D, RowSel* __restrict__ sel,
                                                       double* __restrict__ core) {
    extern __shared__ __align__(16) unsigned char smem[];
    Panels& s = *reinterpret_cast<Panels*>(smem);
    unsigned int(*hist)[BINS] = reinterpret_cast<unsigned int(*)[BINS]>(smem + sizeof(Panels));   // LIST rows: 128 u64 keys
    __shared__ unsigned long long s_prefix[BI], s_mask[BI];
    __shared__ int s_mode[BI], s_shift[BI];
    __shared__ unsigned int s_cnt[BI];
    __shared__ int s_busy;
    const long long row0 = (long long)blockIdx.x * BI;
    if (threadIdx.x == 0) s_busy = 0;
    __syncthreads();
    if (threadIdx.x < BI) {
        const long long i = row0 + threadIdx.x;
        int mode = MODE_DONE;
        if (i < n) {
            const RowSel rs = sel[i];
            mode = rs.mode;
            s_prefix[threadIdx.x] = rs.prefix;
            s_mask[threadIdx.x] = rs.nbits ? ~0ull << (64 - rs.nbits) : 0ull;
            s_shift[threadIdx.x] = 56 - rs.nbits;
        }
        s_mode[threadIdx.x] = mode;
        s_cnt[threadIdx.x] = 0;
        if (mode != MODE_DONE) s_busy = 1;
    }
    for (int e = threadIdx.x; e < BI * BINS; e += NT) hist[e / BINS][e % BINS] = 0;
    __syncthreads();
    if (!s_busy) return;

    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4];
    for (long long col0 = 0; col0 < n; col0 += BJ) {
        sq_tile(x, n, D, row0, col0, s, acc);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int rl = ty + 16 * r;
            const int mode = s_mode[rl];
            if (mode == MODE_DONE) continue;
            const unsigned long long mask = s_mask[rl], prefix = s_prefix[rl];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const unsigned long long key = (unsigned long long)__double_as_longlong(acc[r][c]);
                if (col0 + tx + 16 * c >= n || (key & mask) != prefix) continue;
                if (mode == MODE_HIST) {
                    atomicAdd(&hist[rl][(key >> s_shift[rl]) & (BINS - 1)], 1u);
                } else {
                    const unsigned int slot = atomicAdd(&s_cnt[rl], 1u);
                    if (slot < LIST_MAX) reinterpret_cast<unsigned long long*>(hist[rl])[slot] = key;
                }
            }
        }
    }
    __syncthreads();

    // LIST rows: the rank-th smallest of the collected keys (all threads; keys ordered by (value, slot))
    for (int e = threadIdx.x; e < BI * LIST_MAX; e += NT) {
        const int rl = e / LIST_MAX, m = e % LIST_MAX;
        if (s_mode[rl] != MODE_LIST || m >= (int)s_cnt[rl]) continue;
        const unsigned long long* keys = reinterpret_cast<const unsigned long long*>(hist[rl]);
        const unsigned long long km = keys[m];
        long long before = 0;
        for (int q = 0; q < (int)s_cnt[rl]; ++q) before += keys[q] < km || (keys[q] == km && q < m);
        const long long i = row0 + rl;
        if (before + 1 == sel[i].rank) {
            core[i] = __dsqrt_rn(__longlong_as_double((long long)km));
            sel[i].mode = MODE_DONE;
        }
    }
    // HIST rows: pick the bucket of the rank-th key and narrow the prefix by one digit
    if (threadIdx.x < BI && s_mode[threadIdx.x] == MODE_HIST) {
        const int rl = threadIdx.x;
        const long long i = row0 + rl;
        RowSel rs = sel[i];
        long long below = 0;
        int b = 0;
        for (; b < BINS - 1; ++b) {
            if (below + hist[rl][b] >= rs.rank) break;
            below += hist[rl][b];
        }
        rs.prefix |= (unsigned long long)b << s_shift[rl];
        rs.rank -= below;
        rs.count = hist[rl][b];
        rs.nbits += 8;
        if (rs.nbits == 64) {
            core[i] = __dsqrt_rn(__longlong_as_double((long long)rs.prefix));
            rs.mode = MODE_DONE;
        } else if (rs.count <= LIST_MAX) {
            rs.mode = MODE_LIST;
        }
        sel[i] = rs;
    }
}

// one Borůvka round: for every point the lightest edge (w, min(i, j), max(i, j)) to a point of another component;
// pt_w / pt_pair receive it and comp_w[comp[i]] its weight bits (atomicMin; non-negative doubles order like their bits)
__global__ void __launch_bounds__(NT) mst_nearest_kernel(const float* __restrict__ x, long long n, int D, const double* __restrict__ core,
                                                         const int* __restrict__ comp, unsigned long long* __restrict__ pt_w,
                                                         unsigned long long* __restrict__ pt_pair, unsigned long long* __restrict__ comp_w) {
    __shared__ Panels s;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const long long row0 = (long long)blockIdx.x * BI;
    double ci[4];
    int gi[4];
    unsigned long long bw[4], bp[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const long long i = row0 + ty + 16 * r;
        ci[r] = i < n ? core[i] : 0.0;
        gi[r] = i < n ? comp[i] : -1;
        bw[r] = bp[r] = NONE;
    }
    double acc[4][4];
    for (long long col0 = 0; col0 < n; col0 += BJ) {
        sq_tile(x, n, D, row0, col0, s, acc);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const long long j = col0 + tx + 16 * c;
            if (j >= n) continue;
            const int cj = comp[j];
            const double corej = core[j];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                if (gi[r] < 0 || gi[r] == cj) continue;
                const long long i = row0 + ty + 16 * r;
                const double w = fmax(fmax(ci[r], corej), __dsqrt_rn(acc[r][c]));
                const unsigned long long wb = (unsigned long long)__double_as_longlong(w);
                const unsigned long long pair = i < j ? ((unsigned long long)i << 32) | (unsigned long long)j
                                                      : ((unsigned long long)j << 32) | (unsigned long long)i;
                if (wb < bw[r] || (wb == bw[r] && pair < bp[r])) {
                    bw[r] = wb;
                    bp[r] = pair;
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
        for (int off = 8; off > 0; off >>= 1) {   // the 16 lanes of a row are one half-warp
            const unsigned long long ow = __shfl_xor_sync(0xffffffffu, bw[r], off, 16);
            const unsigned long long op = __shfl_xor_sync(0xffffffffu, bp[r], off, 16);
            if (ow < bw[r] || (ow == bw[r] && op < bp[r])) {
                bw[r] = ow;
                bp[r] = op;
            }
        }
        const long long i = row0 + ty + 16 * r;
        if (tx == 0 && i < n) {
            pt_w[i] = bw[r];
            pt_pair[i] = bp[r];
            if (bw[r] != NONE) atomicMin(&comp_w[gi[r]], bw[r]);
        }
    }
}

// the component's lightest edge: among its points whose edge has the component's lightest weight, the smallest pair
__global__ void mst_pair_kernel(long long n, const int* __restrict__ comp, const unsigned long long* __restrict__ pt_w,
                                const unsigned long long* __restrict__ pt_pair, const unsigned long long* __restrict__ comp_w,
                                unsigned long long* __restrict__ comp_pair) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n || pt_w[i] == NONE) return;
    const int c = comp[i];
    if (pt_w[i] == comp_w[c]) atomicMin(&comp_pair[c], pt_pair[i]);
}

constexpr size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

constexpr size_t CORE_SMEM = sizeof(Panels) + (size_t)BI * BINS * sizeof(unsigned int);
static_assert(LIST_MAX * sizeof(unsigned long long) == BINS * sizeof(unsigned int), "a LIST row reuses its histogram");

struct MstWs {
    int* comp;
    unsigned long long *pt_w, *pt_pair, *comp_w, *comp_pair;
};

size_t core_ws(int64_t n) { return align256((size_t)n * sizeof(RowSel)); }
size_t mst_ws(int64_t n, MstWs* w, char* base) {
    const size_t u = align256((size_t)n * 8), c = align256((size_t)n * 4);
    if (w) {
        w->comp = reinterpret_cast<int*>(base);
        w->pt_w = reinterpret_cast<unsigned long long*>(base + c);
        w->pt_pair = reinterpret_cast<unsigned long long*>(base + c + u);
        w->comp_w = reinterpret_cast<unsigned long long*>(base + c + 2 * u);
        w->comp_pair = reinterpret_cast<unsigned long long*>(base + c + 3 * u);
    }
    return c + 4 * u;
}

constexpr long long MAX_N = 0x7fffffffLL;   // point indices travel as 32-bit halves of a 64-bit pair key

int check_shape(const char* who, int64_t n, int D) {
    if (n < 1 || n > MAX_N) return set_error(IDL_EINVAL, "%s: n must be in 1..2147483647 (got %lld)", who, (long long)n);
    if (D < 1) return set_error(IDL_EINVAL, "%s: D must be >= 1 (got %lld)", who, (long long)D);
    return IDL_OK;
}

int check_ws(const char* who, int64_t n, int D, size_t ws_bytes) {
    const size_t need = idl_hdbscan_workspace_bytes(n, D);
    if (ws_bytes < need) return set_error(IDL_EINVAL, "%s: workspace too small (need %lld bytes)", who, (long long)need);
    return IDL_OK;
}

}  // namespace
}  // namespace idl

using namespace idl;

extern "C" size_t idl_hdbscan_workspace_bytes(int64_t n, int D) {
    if (n < 1 || n > MAX_N || D < 1) return 0;
    return std::max(core_ws(n), mst_ws(n, nullptr, nullptr));
}

extern "C" int idl_core_distances(const float* d_x, int64_t n, int D, int64_t k, double* d_core, void* d_ws, size_t ws_bytes, void* stream) {
    static const char* who = "idl_core_distances";
    if (!d_x || !d_core || !d_ws) return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (int rc = check_shape(who, n, D)) return rc;
    if (k < 1 || k > n) return set_error(IDL_EINVAL, "%s: k must be in 1..n (got %lld)", who, (long long)k);
    if (int rc = check_ws(who, n, D, ws_bytes)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    RowSel* sel = reinterpret_cast<RowSel*>(d_ws);
    IDL_CUDA_CHECK(cudaFuncSetAttribute(core_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CORE_SMEM));
    core_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sel, n, k);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    const unsigned grid = (unsigned)((n + BI - 1) / BI);
    for (int pass = 0; pass < 8; ++pass) {   // every row is done after at most 8 digits; finished CTAs exit at once
        core_pass_kernel<<<grid, NT, CORE_SMEM, st>>>(d_x, n, D, sel, d_core);
        note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
    }
    return IDL_OK;
}

extern "C" int idl_mreach_mst(const float* d_x, const double* d_core, int64_t n, int D, int64_t* d_src, int64_t* d_dst, double* d_w, void* d_ws,
                              size_t ws_bytes, void* stream) {
    static const char* who = "idl_mreach_mst";
    if (!d_x || !d_core || !d_src || !d_dst || !d_w || !d_ws) return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (int rc = check_shape(who, n, D)) return rc;
    if (int rc = check_ws(who, n, D, ws_bytes)) return rc;
    if (n == 1) return IDL_OK;   // no edges
    cudaStream_t st = (cudaStream_t)stream;
    MstWs w;
    mst_ws(n, &w, reinterpret_cast<char*>(d_ws));

    // components are dense ids 0..m-1; the host keeps the point -> component map and merges between rounds
    std::vector<int> comp(n);
    std::iota(comp.begin(), comp.end(), 0);
    std::vector<unsigned long long> cw, cp;
    std::vector<int> parent, newid;
    std::vector<int64_t> src, dst;
    std::vector<double> wt;
    src.reserve(n - 1); dst.reserve(n - 1); wt.reserve(n - 1);
    auto find = [&](int a) {
        while (parent[a] != a) a = parent[a] = parent[parent[a]];
        return a;
    };
    long long m = n;
    const unsigned grid = (unsigned)((n + BI - 1) / BI);
    while (m > 1) {
        IDL_CUDA_CHECK(cudaMemcpyAsync(w.comp, comp.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
        IDL_CUDA_CHECK(cudaMemsetAsync(w.comp_w, 0xff, m * 8, st));
        IDL_CUDA_CHECK(cudaMemsetAsync(w.comp_pair, 0xff, m * 8, st));
        mst_nearest_kernel<<<grid, NT, 0, st>>>(d_x, n, D, d_core, w.comp, w.pt_w, w.pt_pair, w.comp_w);
        note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
        mst_pair_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, w.comp, w.pt_w, w.pt_pair, w.comp_w, w.comp_pair);
        note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
        cw.resize(m);
        cp.resize(m);
        IDL_CUDA_CHECK(cudaMemcpyAsync(cw.data(), w.comp_w, m * 8, cudaMemcpyDeviceToHost, st));
        IDL_CUDA_CHECK(cudaMemcpyAsync(cp.data(), w.comp_pair, m * 8, cudaMemcpyDeviceToHost, st));
        IDL_CUDA_CHECK(cudaStreamSynchronize(st));

        // every component's lightest edge joins it to another; with the strict edge order (w, min, max) the only
        // cycles are two components choosing the same edge, which the union-find skips the second time
        parent.resize(m);
        std::iota(parent.begin(), parent.end(), 0);
        for (long long c = 0; c < m; ++c) {
            if (cw[c] == NONE || cp[c] == NONE) return set_error(IDL_ECUDA, "%s: component without an outgoing edge", who);
            const int64_t a = (int64_t)(cp[c] >> 32), b = (int64_t)(cp[c] & 0xffffffffu);
            const int ra = find(comp[a]), rb = find(comp[b]);
            if (ra == rb) continue;
            parent[std::max(ra, rb)] = std::min(ra, rb);
            src.push_back(a);
            dst.push_back(b);
            double wd;
            memcpy(&wd, &cw[c], sizeof(wd));
            wt.push_back(wd);
        }
        newid.assign(m, -1);
        long long m2 = 0;
        for (long long c = 0; c < m; ++c) {
            const int r = find((int)c);
            if (newid[r] < 0) newid[r] = (int)m2++;
        }
        for (int64_t i = 0; i < n; ++i) comp[i] = newid[find(comp[i])];
        m = m2;
    }
    if ((int64_t)src.size() != n - 1) return set_error(IDL_ECUDA, "%s: spanning tree has %lld edges", who, (long long)src.size());

    // orient every edge away from point 0, parent first, as sklearn's Prim (which grows the tree from point 0) emits it:
    // make_single_linkage takes the (left, right) children of each merge from the edge direction, and the cluster
    // numbering of tree_to_labels follows them
    std::vector<int64_t> off(n + 1, 0), adj(2 * (n - 1)), stack;
    for (int64_t e = 0; e < n - 1; ++e) ++off[src[e] + 1], ++off[dst[e] + 1];
    for (int64_t i = 0; i < n; ++i) off[i + 1] += off[i];
    std::vector<int64_t> fill(off.begin(), off.end() - 1);
    for (int64_t e = 0; e < n - 1; ++e) adj[fill[src[e]]++] = e, adj[fill[dst[e]]++] = e;
    std::vector<char> seen(n, 0);
    seen[0] = 1;
    stack.push_back(0);
    while (!stack.empty()) {
        const int64_t u = stack.back();
        stack.pop_back();
        for (int64_t q = off[u]; q < off[u + 1]; ++q) {
            const int64_t e = adj[q];
            const int64_t v = src[e] == u ? dst[e] : src[e];
            if (seen[v]) continue;
            seen[v] = 1;
            src[e] = u;
            dst[e] = v;
            stack.push_back(v);
        }
    }
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_src, src.data(), (n - 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_dst, dst.data(), (n - 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_w, wt.data(), (n - 1) * sizeof(double), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaStreamSynchronize(st));   // the host vectors die on return
    return IDL_OK;
}
