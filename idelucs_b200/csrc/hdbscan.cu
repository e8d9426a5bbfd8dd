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
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <numeric>
#include <string>
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

__global__ void core_init_kernel(RowSel* __restrict__ sel, long long n, long long k, long long row_begin, long long row_end) {
    const long long i = row_begin + blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < row_end) sel[i] = RowSel{0ull, k, n, 0, n <= LIST_MAX ? MODE_LIST : MODE_HIST};
}

// one radix-select pass: every unfinished row either histograms the next 8-bit digit of the keys that match its prefix
// (MODE_HIST) or collects those keys and picks the rank-th (MODE_LIST).  CTAs whose rows are all done return at once.
// CTA b owns the rows row_begin + 64 b ..; rows at or past row_end are treated as done (their keys are not collected).
__global__ void __launch_bounds__(NT) core_pass_kernel(const float* __restrict__ x, long long n, int D, long long row_begin, long long row_end,
                                                       RowSel* __restrict__ sel, double* __restrict__ core) {
    extern __shared__ __align__(16) unsigned char smem[];
    Panels& s = *reinterpret_cast<Panels*>(smem);
    unsigned int(*hist)[BINS] = reinterpret_cast<unsigned int(*)[BINS]>(smem + sizeof(Panels));   // LIST rows: 128 u64 keys
    __shared__ unsigned long long s_prefix[BI], s_mask[BI];
    __shared__ int s_mode[BI], s_shift[BI];
    __shared__ unsigned int s_cnt[BI];
    __shared__ int s_busy;
    const long long row0 = row_begin + (long long)blockIdx.x * BI;
    if (threadIdx.x == 0) s_busy = 0;
    __syncthreads();
    if (threadIdx.x < BI) {
        const long long i = row0 + threadIdx.x;
        int mode = MODE_DONE;
        if (i < row_end) {
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
// pt_w / pt_pair receive it and comp_w[comp[i]] its weight bits (atomicMin; non-negative doubles order like their bits).
// Only the points i of [row_begin, row_end) are searched from (CTA b owns row_begin + 64 b ..); their partners j are all n.
__global__ void __launch_bounds__(NT) mst_nearest_kernel(const float* __restrict__ x, long long n, int D, long long row_begin, long long row_end,
                                                         const double* __restrict__ core, const int* __restrict__ comp,
                                                         unsigned long long* __restrict__ pt_w, unsigned long long* __restrict__ pt_pair,
                                                         unsigned long long* __restrict__ comp_w) {
    __shared__ Panels s;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const long long row0 = row_begin + (long long)blockIdx.x * BI;
    double ci[4];
    int gi[4];
    unsigned long long bw[4], bp[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const long long i = row0 + ty + 16 * r;
        ci[r] = i < row_end ? core[i] : 0.0;
        gi[r] = i < row_end ? comp[i] : -1;
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
        if (tx == 0 && i < row_end) {
            pt_w[i] = bw[r];
            pt_pair[i] = bp[r];
            if (bw[r] != NONE) atomicMin(&comp_w[gi[r]], bw[r]);
        }
    }
}

// the component's lightest edge: among its points (of [row_begin, row_end)) whose edge has the component's lightest weight,
// the smallest pair
__global__ void mst_pair_kernel(long long row_begin, long long row_end, const int* __restrict__ comp, const unsigned long long* __restrict__ pt_w,
                                const unsigned long long* __restrict__ pt_pair, const unsigned long long* __restrict__ comp_w,
                                unsigned long long* __restrict__ comp_pair) {
    const long long i = row_begin + blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= row_end || pt_w[i] == NONE) return;
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

// the k-th smallest distance of every row of [row_begin, row_end) (arguments already checked; an empty range enqueues nothing)
int core_rows(const float* d_x, int64_t n, int D, int64_t k, int64_t row_begin, int64_t row_end, double* d_core, void* d_ws, cudaStream_t st) {
    const int64_t rows = row_end - row_begin;
    if (rows == 0) return IDL_OK;
    RowSel* sel = reinterpret_cast<RowSel*>(d_ws);
    IDL_CUDA_CHECK(cudaFuncSetAttribute(core_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CORE_SMEM));
    core_init_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(sel, n, k, row_begin, row_end);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    const unsigned grid = (unsigned)((rows + BI - 1) / BI);
    for (int pass = 0; pass < 8; ++pass) {   // every row is done after at most 8 digits; finished CTAs exit at once
        core_pass_kernel<<<grid, NT, CORE_SMEM, st>>>(d_x, n, D, row_begin, row_end, sel, d_core);
        note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
    }
    return IDL_OK;
}

// restores the caller's current device on every return path
struct DeviceGuard {
    int dev = -1;
    ~DeviceGuard() {
        if (dev >= 0) cudaSetDevice(dev);
    }
};

// One Borůvka merge on the host: cw / cp hold every component's lightest outgoing edge (weight bits, pair key).  With the
// strict edge order (w, min, max) the only cycles are two components choosing the same edge, which the union-find skips the
// second time.  The new edges are appended to src / dst / wt, comp is renumbered densely and m becomes the new count.
int merge_round(const char* who, std::vector<int>& comp, const std::vector<unsigned long long>& cw, const std::vector<unsigned long long>& cp,
                long long& m, std::vector<int64_t>& src, std::vector<int64_t>& dst, std::vector<double>& wt) {
    std::vector<int> parent(m), newid(m, -1);
    std::iota(parent.begin(), parent.end(), 0);
    auto find = [&](int a) {
        while (parent[a] != a) a = parent[a] = parent[parent[a]];
        return a;
    };
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
    long long m2 = 0;
    for (long long c = 0; c < m; ++c) {
        const int r = find((int)c);
        if (newid[r] < 0) newid[r] = (int)m2++;
    }
    for (size_t i = 0; i < comp.size(); ++i) comp[i] = newid[find(comp[i])];
    m = m2;
    return IDL_OK;
}

// orient every edge of the spanning tree away from point 0, parent first, as sklearn's Prim (which grows the tree from point
// 0) emits it: make_single_linkage takes the (left, right) children of each merge from the edge direction, and the cluster
// numbering of tree_to_labels follows them
void orient_from_point0(int64_t n, std::vector<int64_t>& src, std::vector<int64_t>& dst) {
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
}

// The mutual-reachability MST with its all-pairs work split into row ranges that partition [0, n) (arguments already checked,
// n >= 2).  Part p searches the lightest outgoing edge of the points of its rows on devices[p], with its own replica of x and
// core, its own workspace and streams[p].  Components are dense ids 0..m-1; the host keeps the point -> component map,
// reduces the parts' per-component minima and merges the components between rounds.
int mst_parts(const char* who, int n_parts, const int* devices, const float* const* d_x, const double* const* d_core, const int64_t* row_begin,
              const int64_t* row_end, int64_t n, int D, int64_t* d_src, int64_t* d_dst, double* d_w, void* const* d_ws, void* const* streams) {
    DeviceGuard guard;
    IDL_CUDA_CHECK(cudaGetDevice(&guard.dev));
    std::vector<MstWs> w(n_parts);
    for (int p = 0; p < n_parts; ++p) mst_ws(n, &w[p], reinterpret_cast<char*>(d_ws[p]));
    std::vector<int> comp(n);
    std::iota(comp.begin(), comp.end(), 0);
    std::vector<std::vector<unsigned long long>> pw(n_parts), pp(n_parts);
    std::vector<unsigned long long> cw, cp;
    std::vector<int64_t> src, dst;
    std::vector<double> wt;
    src.reserve(n - 1); dst.reserve(n - 1); wt.reserve(n - 1);
    long long m = n;
    while (m > 1) {
        // every part is launched before any is read back: a copy to pageable memory blocks the host until its stream is done
        for (int p = 0; p < n_parts; ++p) {
            const int64_t rows = row_end[p] - row_begin[p];
            if (rows == 0) continue;
            cudaStream_t st = (cudaStream_t)streams[p];
            IDL_CUDA_CHECK(cudaSetDevice(devices[p]));
            IDL_CUDA_CHECK(cudaMemcpyAsync(w[p].comp, comp.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
            IDL_CUDA_CHECK(cudaMemsetAsync(w[p].comp_w, 0xff, m * 8, st));
            IDL_CUDA_CHECK(cudaMemsetAsync(w[p].comp_pair, 0xff, m * 8, st));
            mst_nearest_kernel<<<(unsigned)((rows + BI - 1) / BI), NT, 0, st>>>(d_x[p], n, D, row_begin[p], row_end[p], d_core[p], w[p].comp,
                                                                               w[p].pt_w, w[p].pt_pair, w[p].comp_w);
            note_launch();
            IDL_CUDA_CHECK(cudaGetLastError());
            mst_pair_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(row_begin[p], row_end[p], w[p].comp, w[p].pt_w, w[p].pt_pair,
                                                                           w[p].comp_w, w[p].comp_pair);
            note_launch();
            IDL_CUDA_CHECK(cudaGetLastError());
        }
        for (int p = 0; p < n_parts; ++p) {
            if (row_end[p] == row_begin[p]) continue;
            cudaStream_t st = (cudaStream_t)streams[p];
            pw[p].resize(m);
            pp[p].resize(m);
            IDL_CUDA_CHECK(cudaSetDevice(devices[p]));
            IDL_CUDA_CHECK(cudaMemcpyAsync(pw[p].data(), w[p].comp_w, m * 8, cudaMemcpyDeviceToHost, st));
            IDL_CUDA_CHECK(cudaMemcpyAsync(pp[p].data(), w[p].comp_pair, m * 8, cudaMemcpyDeviceToHost, st));
            IDL_CUDA_CHECK(cudaStreamSynchronize(st));
        }
        // per component the lexicographic minimum of (w, pair) over the parts: what the two atomicMin steps give on one device
        cw.assign(m, NONE);
        cp.assign(m, NONE);
        for (int p = 0; p < n_parts; ++p) {
            if (row_end[p] == row_begin[p]) continue;
            for (long long c = 0; c < m; ++c)
                if (pw[p][c] < cw[c] || (pw[p][c] == cw[c] && pp[p][c] < cp[c])) cw[c] = pw[p][c], cp[c] = pp[p][c];
        }
        if (int rc = merge_round(who, comp, cw, cp, m, src, dst, wt)) return rc;
    }
    if ((int64_t)src.size() != n - 1) return set_error(IDL_ECUDA, "%s: spanning tree has %lld edges", who, (long long)src.size());
    orient_from_point0(n, src, dst);
    cudaStream_t st = (cudaStream_t)streams[0];
    IDL_CUDA_CHECK(cudaSetDevice(devices[0]));
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_src, src.data(), (n - 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_dst, dst.data(), (n - 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaMemcpyAsync(d_w, wt.data(), (n - 1) * sizeof(double), cudaMemcpyHostToDevice, st));
    IDL_CUDA_CHECK(cudaStreamSynchronize(st));   // the host vectors die on return
    return IDL_OK;
}

}  // namespace

int check_rows(const char* who, int64_t n, int64_t row_begin, int64_t row_end) {
    if (row_begin < 0 || row_begin > row_end || row_end > n) {
        char what[160];
        snprintf(what, sizeof(what), "%s: row range [%lld, %lld) is not inside [0, %lld)", who, (long long)row_begin, (long long)row_end,
                 (long long)n);
        return set_error(IDL_EINVAL, "%s", what);
    }
    return IDL_OK;
}

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
    return core_rows(d_x, n, D, k, 0, n, d_core, d_ws, (cudaStream_t)stream);
}

extern "C" int idl_core_distances_rows(const float* d_x, int64_t n, int D, int64_t k, int64_t row_begin, int64_t row_end, double* d_core,
                                       void* d_ws, size_t ws_bytes, void* stream) {
    static const char* who = "idl_core_distances_rows";
    if (!d_x || !d_core || !d_ws) return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (int rc = check_shape(who, n, D)) return rc;
    if (k < 1 || k > n) return set_error(IDL_EINVAL, "%s: k must be in 1..n (got %lld)", who, (long long)k);
    if (int rc = check_rows(who, n, row_begin, row_end)) return rc;
    if (int rc = check_ws(who, n, D, ws_bytes)) return rc;
    return core_rows(d_x, n, D, k, row_begin, row_end, d_core, d_ws, (cudaStream_t)stream);
}

extern "C" int idl_mreach_mst(const float* d_x, const double* d_core, int64_t n, int D, int64_t* d_src, int64_t* d_dst, double* d_w, void* d_ws,
                              size_t ws_bytes, void* stream) {
    static const char* who = "idl_mreach_mst";
    if (!d_x || !d_core || !d_src || !d_dst || !d_w || !d_ws) return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (int rc = check_shape(who, n, D)) return rc;
    if (int rc = check_ws(who, n, D, ws_bytes)) return rc;
    if (n == 1) return IDL_OK;   // no edges
    int dev;
    IDL_CUDA_CHECK(cudaGetDevice(&dev));
    const int64_t begin = 0;
    return mst_parts(who, 1, &dev, &d_x, &d_core, &begin, &n, n, D, d_src, d_dst, d_w, &d_ws, &stream);
}

extern "C" int idl_mreach_mst_parts(int n_parts, const int* devices, const float* const* d_x, const double* const* d_core, const int64_t* row_begin,
                                    const int64_t* row_end, int64_t n, int D, int64_t* d_src, int64_t* d_dst, double* d_w, void* const* d_ws,
                                    const size_t* ws_bytes, void* const* streams) {
    static const char* who = "idl_mreach_mst_parts";
    if (!devices || !d_x || !d_core || !row_begin || !row_end || !d_src || !d_dst || !d_w || !d_ws || !ws_bytes || !streams)
        return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (n_parts < 1) return set_error(IDL_EINVAL, "%s: n_parts must be >= 1 (got %lld)", who, (long long)n_parts);
    std::vector<std::string> part(n_parts);   // "idl_mreach_mst_parts: part p", the prefix of a part's error texts
    for (int p = 0; p < n_parts; ++p) part[p] = std::string(who) + ": part " + std::to_string(p);
    for (int p = 0; p < n_parts; ++p)
        if (!d_x[p] || !d_core[p] || !d_ws[p]) return set_error(IDL_EINVAL, "%s: null pointer", part[p].c_str());
    if (int rc = check_shape(who, n, D)) return rc;
    for (int p = 0; p < n_parts; ++p)
        if (int rc = check_rows(part[p].c_str(), n, row_begin[p], row_end[p])) return rc;
    for (int p = 0; p <= n_parts; ++p) {   // part p begins where part p - 1 ends; part 0 at 0, and the last part ends at n
        const int64_t at = p < n_parts ? row_begin[p] : n, want = p ? row_end[p - 1] : 0;
        if (at == want) continue;
        char what[200];
        snprintf(what, sizeof(what), "%s: the row ranges do not partition [0, %lld) in order: part %d %s at %lld, not %lld", who, (long long)n,
                 p < n_parts ? p : p - 1, p < n_parts ? "begins" : "ends", (long long)(p < n_parts ? at : want), (long long)(p < n_parts ? want : at));
        return set_error(IDL_EINVAL, "%s", what);
    }
    for (int p = 0; p < n_parts; ++p)
        if (int rc = check_ws(part[p].c_str(), n, D, ws_bytes[p])) return rc;
    if (n == 1) return IDL_OK;   // no edges
    return mst_parts(who, n_parts, devices, d_x, d_core, row_begin, row_end, n, D, d_src, d_dst, d_w, d_ws, streams);
}
