// idelucs_b200 — sm_100a kernels K1 (pack), K2/K3 (k-mer profile + mimic variants), K4 (scaler)
// and the C ABI of include/idelucs_b200.h for them.  K5 (IIC loss) lives in train_ops.cu.
//
// Design (DESIGN.md §4): one CTA owns one sequence at a time.  It builds the CLEAN 4^k
// histogram once in shared memory (rolling k-mer index from 2-bit packed bases read with
// 128-bit loads, shared-memory atomics, no global atomics).  Every mimic variant is then
// produced by patching that histogram with the +-1 deltas of the k windows around each
// mutated base (mutations come from a counter-based Philox RNG in registers, or from an
// explicit edit list), streaming the normalised / standardised profile to HBM with 128-bit
// streaming stores, and un-patching.  Mutated sequences never exist in memory; the path is
// bound by the HBM write of the profiles.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/idelucs_b200.h"
#include "core.cuh"
#include "common.h"

namespace idl {

// ---------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, const char* a, long long b) {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}

static std::atomic<long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

constexpr int LIST_CAP = 2048;   // on-chip edit list entries per CTA
constexpr int CH_MIN_LEN = 65536; // items at least this long take the chunked path (chunked.cuh) when the caller provides its scratch
constexpr int SG = 32;           // variant slots per supergroup (Random_N removals precomputed together)
constexpr int REM_CAP = 3840;    // removed k-mers buffered per supergroup (32 slots x 20 draws x k=6)
constexpr int ENT_CAP = 1024;    // Random_N draws buffered per supergroup (aliases the edit list)
constexpr int SSEQ_CHUNKS = 320; // sequences up to 20480 bases are staged in shared memory (codes + mask)
constexpr int SSEQ_CW = SSEQ_CHUNKS * 4 + 4, SSEQ_MW = SSEQ_CHUNKS * 2 + 2;
constexpr int SVARS = 64;        // variant descriptors cached in shared memory
constexpr int STABS = 4;         // gap tables cached in shared memory

struct VarDesc {
    int32_t kind, rng_id, n_bp, explicit_idx, tab1, tab2;
    float slope1, slope2;
};

// launch plan passed BY VALUE as a kernel parameter (no host->device copy, nothing cached between calls, CUDA-graph
// capture records it with the launch): the variant descriptors, output offsets and gap tables of calls with at most SVARS
// variants / slots and STABS distinct mutation rates.  Bigger plans are uploaded into the workspace instead.
struct Plan {
    VarDesc vars[SVARS];
    long long out_off[SVARS];
    uint32_t gtab[STABS][RNG_BLOCK];
};

struct ProfParams {
    const uint32_t* codes;
    const uint32_t* nmask;
    const int64_t* chunk_off;
    const int32_t* len;
    const int32_t* sidx;
    const int32_t* sel;
    long long n_items, seq_id0, n_seqs_total;
    int S, n_vars, n_tabs;
    const VarDesc* vars;
    unsigned long long seed;
    const uint32_t* gtab;
    const int64_t* edit_off;
    const uint32_t* edits;
    void* out;
    const int64_t* out_off;
    long long out_stride;
    int pseudocount, accumulate;
    int cta_cap;                      // host side: at most this many CTAs per SM for the generic kernel (0 = as many as fit)
    const float* mean;
    const float* scale;
    const float* rscale;  // 1/scale (IEEE), computed into the workspace by rscale_kernel
    int32_t* status;
    unsigned long long* work_counter;
    int only_deferred;                // generic kernel: redo only the items the producer/consumer kernel flagged (status bit 1)
    double* stats_partials;           // OUT_STATS: per-CTA (mean, M2) [gridDim][2][4^k]
    double* stats_n;                  // OUT_STATS: per-CTA row count [gridDim]
    int inline_plan;                  // descriptors / offsets / tables come from the Plan kernel parameter (else from vars / out_off / gtab)
    void* prep;                       // prepared buffer (prep.cuh): written by prep_kernel, read by colstats16 / the producer/consumer kernel
    unsigned long long prep_stamp;    // what the prepared buffer must have been prepared for
    const int* long_overflow;         // chunked path active (chunked.cuh): items of >= CH_MIN_LEN bases are skipped here while *long_overflow == 0
};
static_assert(sizeof(ProfParams) + sizeof(Plan) <= 4000, "kernel parameters must stay below the 4 KB limit");

constexpr int OUT_STATS = 4;          // internal out kind: column statistics of slot 0's float32 frequencies, nothing is written per row

// ---------------------------------------------------------------------------------------
// K1 pack
// ---------------------------------------------------------------------------------------
constexpr int PACK_NT = 256;

__global__ void __launch_bounds__(PACK_NT) pack_kernel(const uint8_t* __restrict__ ascii,
                                                        const int64_t* __restrict__ byte_off,
                                                        const int64_t* __restrict__ chunk_off, long long n, int strict,
                                                        uint32_t* __restrict__ codes, uint32_t* __restrict__ nmask,
                                                        int32_t* __restrict__ len, unsigned long long* __restrict__ bad) {
    // byte -> class table of the alphabet (core.cuh base_class: the switch itself costs ~40 divergent instructions per byte):
    // bits 0-1 = code (0 for a non-base), bit 2 = reset flag, bits 3-5 = class when the byte is deleted / invalid (5 / 6), else 0
    __shared__ uint8_t lut[256];
    for (int i = threadIdx.x; i < 256; i += PACK_NT) {
        const uint32_t cls = base_class((uint32_t)i, strict);
        lut[i] = (uint8_t)(cls < 4 ? cls : (4u | (cls >= 5 ? cls << 3 : 0u)));
    }
    __syncthreads();
    for (long long s = blockIdx.x; s <= n; s += gridDim.x) {
        if (s == n) {  // slack chunk behind the last sequence: all padding
            if (blockIdx.y == 0 && threadIdx.x < 4) codes[chunk_off[n] * 4 + threadIdx.x] = 0u;
            if (blockIdx.y == 0 && threadIdx.x < 2) nmask[chunk_off[n] * 2 + threadIdx.x] = 0xFFFFFFFFu;
            continue;
        }
        const long long b0 = byte_off[s];
        const long long L = byte_off[s + 1] - b0;
        const long long c0 = chunk_off[s];
        const long long nhalf = (chunk_off[s + 1] - c0) * 2;  // 32-base half chunks
        if (blockIdx.y == 0 && threadIdx.x == 0) len[s] = (int32_t)L;
        unsigned long long first_bad = ~0ull;
        for (long long h = (long long)blockIdx.y * PACK_NT + threadIdx.x; h < nhalf; h += (long long)PACK_NT * gridDim.y) {
            // the 32 bytes of the half chunk as 8 little-endian words (padding behind the end of the sequence reads as 'N').  A half
            // chunk that lies completely inside the sequence is read as aligned 32-bit words (every word holds at least one byte of the
            // sequence, so it lies inside the caller's allocation) realigned with funnel shifts: 9 loads instead of 32 byte loads
            // (lanes are 32 bytes apart: every load instruction costs one L1 wavefront per lane)
            uint32_t wv[8];
            long long avail32 = L - h * 32;
            avail32 = avail32 < 0 ? 0 : (avail32 > 32 ? 32 : avail32);
            if (avail32 == 32) {
                const uint8_t* a = ascii + b0 + h * 32;
                const uint32_t sh = ((uint32_t)(uintptr_t)a & 3u) * 8u;
                const uint32_t* a4 = reinterpret_cast<const uint32_t*>(a - ((uintptr_t)a & 3u));
                uint32_t w9[9];
#pragma unroll
                for (int i = 0; i < 8; ++i) w9[i] = __ldg(a4 + i);
                w9[8] = sh ? __ldg(a4 + 8) : 0u;
#pragma unroll
                for (int i = 0; i < 8; ++i) wv[i] = __funnelshift_r(w9[i], w9[i + 1], sh);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    uint32_t w = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) w |= (uint32_t)(i * 4 + j < avail32 ? __ldg(ascii + b0 + h * 32 + i * 4 + j) : (uint8_t)'N') << (8 * j);
                    wv[i] = w;
                }
            }
            uint32_t mw = 0;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                uint32_t cw = 0, m16 = 0, badv = 0;
                int bj = 16;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    uint32_t v = lut[(wv[t * 4 + (j >> 2)] >> (8 * (j & 3))) & 0xFFu];
                    if (t * 16 + j >= avail32) v = 4u;                      // padding: reset, never "bad"
                    if ((v >> 3) && bj == 16) { bj = j; badv = v >> 3; }   // first deleted (5) / invalid (6) byte of this word
                    cw = (cw << 2) | (v & 3u);
                    m16 = (m16 << 1) | ((v >> 2) & 1u);
                }
                codes[c0 * 4 + h * 2 + t] = cw;
                mw = (mw << 16) | m16;
                if (bj < 16) {
                    const unsigned long long v = ((unsigned long long)(h * 32 + t * 16 + bj) << 3) | (unsigned long long)badv;
                    first_bad = v < first_bad ? v : first_bad;
                }
            }
            nmask[c0 * 2 + h] = mw;
        }
        if (first_bad != ~0ull) atomicMin(bad + s, first_bad);
    }
}

// ---------------------------------------------------------------------------------------
// block helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// exclusive scan of one int per thread over the CTA; returns the prefix, *total = CTA sum.
// scratch: NT/32 + 1 ints of shared memory.  Contains two __syncthreads.
template <int NT>
__device__ __forceinline__ int block_exscan(int v, int* scratch, int* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) scratch[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int w = lane < NT / 32 ? scratch[lane] : 0;
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < NT / 32) scratch[lane] = winc - w;
        if (lane == 31) scratch[NT / 32] = winc;
    }
    __syncthreads();
    *total = scratch[NT / 32];
    return scratch[wid] + inc - v;
}

// ---------------------------------------------------------------------------------------
// canonical (reverse-complement folded) rows: IDL_OUT_CANON_* = 8 + the matching frequency kind
// ---------------------------------------------------------------------------------------
constexpr int OUT_CANON_BIT = 8;
constexpr bool is_canon(int out) { return (out & OUT_CANON_BIT) != 0; }

// utils.py:191-206: index of the reverse complement of k-mer m
constexpr uint32_t revcomp_index(uint32_t m, int k) {
    uint32_t x = ~m & ((k < 16 ? (1u << (2 * k)) : 0u) - 1u), r = 0;
    for (int t = 0; t < k; ++t) { r = (r << 2) | (x & 3u); x >>= 2; }
    return r;
}
constexpr int canonical_count(int k) {
    int R = 0;
    for (uint32_t m = 0; m < (1u << (2 * k)); ++m) R += m <= revcomp_index(m, k) ? 1 : 0;
    return R;
}
// the canonical k-mers of idl_revcomp_canonical (kmer <= revcomp, increasing), entry = kmer | revcomp << 16; built by the
// compiler into the module's global data (8.3 KB at k = 6)
template <int K>
struct CanonTab {
    static constexpr int R = canonical_count(K);
    uint32_t e[R];
    constexpr CanonTab() : e{} {
        int r = 0;
        for (uint32_t m = 0; m < (1u << (2 * K)); ++m) {
            const uint32_t c = revcomp_index(m, K);
            if (m <= c) e[r++] = m | (c << 16);
        }
    }
};
template <int K>
__device__ const CanonTab<K> g_canon = CanonTab<K>();

// One canonical row, CTA-wide (contains barriers: every thread of the CTA calls it).  cnt(m) = count of k-mer m plus the
// pseudocount, read from shared memory.  f_r = int((a + b) * 0.5) over the pair (m_r, revcomp(m_r)) (revcomp_fold_kernel's
// rule), T = the exact integer sum of the f_r (a reduction before the first store), then normalize_counts_kernel's float64
// division; the float32 kinds round that quotient and the standardised kind applies idl_standardize_f32's IEEE
// (x - mean32) / scale32.  A thread stores columns r = tid + j NT: scalar, coalesced, any offset and stride.
template <int K, int NT, int OUT, class Cnt>
__device__ __forceinline__ void emit_canon_row(void* out_row, Cnt cnt, const float* mean, const float* scale, int* scan) {
    constexpr int R = CanonTab<K>::R, RPT = (R + NT - 1) / NT;
    int f[RPT];
    int part = 0;
#pragma unroll
    for (int j = 0; j < RPT; ++j) {
        const int r = threadIdx.x + j * NT;
        f[j] = 0;
        if (R % NT == 0 || r < R) {
            const uint32_t e = __ldg(&g_canon<K>.e[r]);
            f[j] = (int)((double)(cnt(e & 0xFFFFu) + cnt(e >> 16)) * 0.5);
            part += f[j];
        }
    }
    int total;
    block_exscan<NT>(part, scan, &total);
    const double dt = (double)total;
#pragma unroll
    for (int j = 0; j < RPT; ++j) {
        const int r = threadIdx.x + j * NT;
        if (R % NT != 0 && r >= R) break;
        const double q = (double)f[j] / dt;
        if (OUT == IDL_OUT_CANON_F64) {
            __stcs(reinterpret_cast<double*>(out_row) + r, q);
        } else {
            float x = (float)q;
            if (OUT == IDL_OUT_CANON_STD_F32) x = (x - __ldg(mean + r)) / __ldg(scale + r);
            __stcs(reinterpret_cast<float*>(out_row) + r, x);
        }
    }
}

// ---------------------------------------------------------------------------------------
// K2/K3 profiles kernel
//
// Per work item (one sequence) a CTA
//   1. counts the clean histogram into hist[] (int32, shared-memory atomics);
//   2. SHORT path (L <= 65535, every count fits 16 bits): keeps G private uint16 copies of
//      the histogram.  Variant slots are consumed G at a time: the copies are patched with
//      the slots' +-1 deltas (Random_N slots by one warp each, concurrently; Bernoulli /
//      explicit slots by the whole CTA), ONE barrier, all threads stream the G profiles
//      (fixed thread <-> bin mapping, scaler statistics in registers, 128-bit streaming
//      stores), ONE barrier, the copies are restored.  Two barriers per G variants.
//   3. LONG path (L > 65535): patches hist[] itself, one variant at a time (int32 counts).
// ---------------------------------------------------------------------------------------
template <int K, int NT>
struct ProfCfg {
    static constexpr int F = 1 << (2 * K);
    static constexpr int VEC = F / 4;                       // 4-bin granules per profile
    static constexpr int VPT = (VEC + NT - 1) / NT;         // granules per thread
    static constexpr int G = (NT / 32) < 8 ? (NT / 32) : 8; // private copies (= variants per barrier pair)
    static constexpr int PRIVW = F / 2 > 2 ? F / 2 : 2;     // words per private copy
    static constexpr int PT = (G * PRIVW) > LIST_CAP ? (G * PRIVW) : LIST_CAP;
};

template <int K, int NT>
struct ProfSmem {
    using C = ProfCfg<K, NT>;
    int hist[C::F];
    uint32_t privtmp[C::PT];          // short path: G private uint16 copies; long path: unsorted Random_N draws
    uint32_t list[LIST_CAP + 8];      // CTA-wide position-sorted edit list; also the supergroup's Random_N draws
    uint32_t sseq[SSEQ_CW + SSEQ_MW]; // packed bases + reset mask of the current sequence (when it fits)
    uint16_t rem[REM_CAP];            // k-mers of the clean windows each Random_N slot removes
    uint32_t gtabs[STABS][RNG_BLOCK]; // geometric gap tables (first STABS of the launch)
    int pre_kind[SG];                 // per slot of the supergroup: 0 none, 1 small Random_N, 2 Bernoulli, 3 other CTA-wide
    int pre_off[SG];                  // first draw of the slot in ent[] (x K = first entry in rem[])
    int pre_nbp[SG];                  // draws of the slot
    int dtot[SG];                     // change of the counted-window total of the slot
    float2 gy[SG];                    // per slot: (float total, 1/total)
    long long grow[SG];               // per slot: byte offset of the output row
    int seg_off[C::G + 1];            // joint Bernoulli pass: list segment of each Bernoulli slot
    unsigned mask_bern, mask_other;   // ballot masks over the supergroup's slots
    int sg_n;                         // slots in the current supergroup
    int sg_ent;                       // Random_N draws in the current supergroup
    int scan[NT / 32 + 2];
    int nvalid;
    long long item;
    unsigned dqmask[NT / 32];         // deferred mode: which of the NT items examined last are flagged
    VarDesc svars[SVARS];             // descriptor cache (first SVARS variants)
    long long sout_off[SVARS];
};

// convert 4 packed uint16 counts (+pc) to exact floats: 2^23 + c is exact for c < 2^23, and
// subtracting 2^23 - pc leaves c + pc exactly (no I2F on the conversion pipe)
__device__ __forceinline__ void cvt4_u16(uint2 pk, float magic, float (&f)[4]) {
    f[0] = __uint_as_float(__byte_perm(pk.x, 0x4B000000u, 0x7410)) - magic;
    f[1] = __uint_as_float(__byte_perm(pk.x, 0x4B000000u, 0x7432)) - magic;
    f[2] = __uint_as_float(__byte_perm(pk.y, 0x4B000000u, 0x7410)) - magic;
    f[3] = __uint_as_float(__byte_perm(pk.y, 0x4B000000u, 0x7432)) - magic;
}

// one 4-bin granule of one profile row.  ci = integer counts INCLUDING the pseudocount
// (COUNTS / F64 / big totals), cf = the same as exact floats (F32 kinds).
template <int OUT>
__device__ __forceinline__ void emit_granule(void* out_row, int vec, const int (&ci)[4], const float (&cf)[4], int total,
                                             float ft, float y, bool big, int accumulate, const float (&mean)[4],
                                             const float (&scale)[4], const float (&rscale)[4]) {
    if (OUT == IDL_OUT_COUNTS_I32) {
        int4* dst = reinterpret_cast<int4*>(out_row) + vec;
        int4 o = make_int4(ci[0], ci[1], ci[2], ci[3]);
        if (accumulate) { const int4 prev = *dst; o.x += prev.x; o.y += prev.y; o.z += prev.z; o.w += prev.w; }
        *dst = o;
    } else if (OUT == IDL_OUT_FREQ_F64) {
        double2* dst = reinterpret_cast<double2*>(out_row) + 2 * vec;
        const double dt = (double)total;
        __stcs(dst, make_double2((double)ci[0] / dt, (double)ci[1] / dt));
        __stcs(dst + 1, make_double2((double)ci[2] / dt, (double)ci[3] / dt));
    } else {
        float q[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            // float32(count/total): for count,total < 2^24 the correctly rounded float division is
            // exactly the reference's float64 division followed by astype(float32) (DESIGN.md §5)
            q[e] = big ? (float)((double)ci[e] / (double)total) : div_rn(cf[e], ft, y);
            if (OUT == IDL_OUT_STD_F32) q[e] = div_rn(q[e] - mean[e], scale[e], rscale[e]);
        }
        __stcs(reinterpret_cast<float4*>(out_row) + vec, make_float4(q[0], q[1], q[2], q[3]));
    }
}

// Blackwell packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2, sm_100+): IEEE round-to-nearest per
// lane, so the results are bit-identical to the scalar path at half the issue slots.
struct Stats2 {           // scaler statistics of one 4-bin granule, ready for the packed ops
    float2 nm01, nm23;    // -mean
    float2 ns01, ns23;    // -scale
    float2 rs01, rs23;    // RN(1/scale)
};
__device__ __forceinline__ Stats2 load_stats2(const float* mean, const float* scale, const float* rscale, int vec, bool on) {
    Stats2 s;
    s.nm01 = s.nm23 = make_float2(0.f, 0.f);
    s.ns01 = s.ns23 = make_float2(-1.f, -1.f);
    s.rs01 = s.rs23 = make_float2(1.f, 1.f);
    if (on) {
        const float4 m = __ldg(reinterpret_cast<const float4*>(mean) + vec);
        const float4 sc = __ldg(reinterpret_cast<const float4*>(scale) + vec);
        const float4 rs = __ldg(reinterpret_cast<const float4*>(rscale) + vec);
        s.nm01 = make_float2(-m.x, -m.y); s.nm23 = make_float2(-m.z, -m.w);
        s.ns01 = make_float2(-sc.x, -sc.y); s.ns23 = make_float2(-sc.z, -sc.w);
        s.rs01 = make_float2(rs.x, rs.y); s.rs23 = make_float2(rs.z, rs.w);
    }
    return s;
}
// one granule: 4 packed uint16 counts -> float32(count+pc)/total [-> standardised] -> one 128-bit streaming store.
// fy = (total, RN(1/total)); same arithmetic as div_rn (core.cuh), two lanes per instruction.
template <bool STD>
__device__ __forceinline__ void emit_granule_u16x2(void* out_row, int vec, uint2 pk, float magic, float2 fy, const Stats2& st) {
    const float2 nmag = make_float2(-magic, -magic), yy = make_float2(fy.y, fy.y), nt = make_float2(-fy.x, -fy.x);
    float2 c01 = make_float2(__uint_as_float(__byte_perm(pk.x, 0x4B000000u, 0x7410)), __uint_as_float(__byte_perm(pk.x, 0x4B000000u, 0x7432)));
    float2 c23 = make_float2(__uint_as_float(__byte_perm(pk.y, 0x4B000000u, 0x7410)), __uint_as_float(__byte_perm(pk.y, 0x4B000000u, 0x7432)));
    c01 = __fadd2_rn(c01, nmag); c23 = __fadd2_rn(c23, nmag);                    // exact count + pseudocount
    float2 q01 = __fmul2_rn(c01, yy), q23 = __fmul2_rn(c23, yy);
    const float2 r01 = __ffma2_rn(q01, nt, c01), r23 = __ffma2_rn(q23, nt, c23);
    q01 = __ffma2_rn(r01, yy, q01); q23 = __ffma2_rn(r23, yy, q23);             // RN(count / total)
    if (STD) {
        const float2 d01 = __fadd2_rn(q01, st.nm01), d23 = __fadd2_rn(q23, st.nm23);
        const float2 t01 = __fmul2_rn(d01, st.rs01), t23 = __fmul2_rn(d23, st.rs23);
        const float2 e01 = __ffma2_rn(t01, st.ns01, d01), e23 = __ffma2_rn(t23, st.ns23, d23);
        q01 = __ffma2_rn(e01, st.rs01, t01); q23 = __ffma2_rn(e23, st.rs23, t23);   // RN((q - mean) / scale)
    }
    __stcs(reinterpret_cast<float4*>(out_row) + vec, make_float4(q01.x, q01.y, q23.x, q23.y));
}

// ---- register-hungry, rarely executed pieces are kept out of line so that the streaming
// ---- loop keeps its scaler statistics in registers (64-register budget at 2 CTAs/SM) ----
struct ItemCtx {
    const uint32_t* codes;
    const uint32_t* nmask;
    int L;
    uint32_t seq_id;
    unsigned long long seed;
};

// patch a private uint16 copy (two counts per word) with the deltas of list entry i
__device__ __forceinline__ void upd16(uint32_t* privc, uint32_t kmer, int d) {
    uint32_t* w = privc + (kmer >> 1);
    const uint32_t inc = 1u << ((kmer & 1u) * 16u);
    if (d > 0) atomicAdd(w, inc); else atomicSub(w, inc);
}
template <int K>
__device__ __noinline__ int apply_priv(const ItemCtx& cx, const uint32_t* list, int n, int i, uint32_t* privc) {
    return apply_entry<K>(cx.codes, cx.nmask, cx.L, list, n, i, [&](uint32_t kmer, int dd) { upd16(privc, kmer, dd); });
}
template <int K>
__device__ __noinline__ int apply_hist(const ItemCtx& cx, const uint32_t* list, int n, int i, int* hist, int sgn) {
    return apply_entry<K>(cx.codes, cx.nmask, cx.L, list, n, i, [&](uint32_t kmer, int dd) { atomicAdd(&hist[kmer], sgn * dd); });
}

template <int K, int NT>
__device__ __forceinline__ const uint32_t* gap_table(const ProfSmem<K, NT>& sm, const ProfParams& p, int t) {
    return t < STABS ? sm.gtabs[t] : p.gtab + t * RNG_BLOCK;
}

// CTA-wide generation of the Bernoulli edit list of the blocks [b_lo, b_hi) (at most NT of them: thread <-> block, mask
// generator) into sm.list, position-sorted; returns the number of entries, or -1 when they do not fit LIST_CAP (nothing
// is written then: the caller retries with fewer blocks — three blocks always fit).  Contains barriers; every thread of
// the CTA must call it.
template <int K, int NT>
__device__ __noinline__ int bern_span(ProfSmem<K, NT>& sm, const ProfParams& p, const ItemCtx& cx, const VarDesc& vd, int b_lo, int b_hi) {
    const int b = b_lo + (int)threadIdx.x;
    BlockMasks m;
    m.a = m.b = m.ch = 0;
    if (b < b_hi)
        m = block_masks(vd.kind, cx.seed, cx.seq_id, (uint32_t)vd.rng_id, b, cx.L, cx.nmask, gap_table(sm, p, vd.tab1), vd.slope1,
                        gap_table(sm, p, vd.tab2), vd.slope2);
    int total;
    const int off = block_exscan<NT>(block_masks_count(m), sm.scan, &total);
    if (total > LIST_CAP) return -1;   // uniform
    block_masks_write(m, b, cx.codes, sm.list + off);
    __syncthreads();
    return total;
}

// Bernoulli slot, any length: tiles of `span` owned blocks plus one context block on each side (an edit's windows only
// involve edits within K-1 positions); fn(total, lo, hi) is called CTA-wide per tile and applies the entries of sm.list whose
// position lies in [lo, hi).  The span halves whenever a tile's edits overflow the on-chip list, so no rate can drop edits.
template <int K, int NT, class Fn>
__device__ __forceinline__ void bern_tiles(ProfSmem<K, NT>& sm, const ProfParams& p, const ItemCtx& cx, const VarDesc& vd, int nblocks, Fn fn) {
    int span = NT - 2;
    for (int tb0 = 0; tb0 < nblocks;) {
        const int t1 = tb0 + span < nblocks ? tb0 + span : nblocks;
        const int total = bern_span<K, NT>(sm, p, cx, vd, tb0 > 0 ? tb0 - 1 : 0, t1 + 1 < nblocks ? t1 + 1 : nblocks);
        if (total < 0) { span = span > 1 ? span >> 1 : 1; continue; }   // (bern_span ends with the barrier that lets the list be rewritten)
        fn(total, tb0 * RNG_BLOCK, (long long)t1 * RNG_BLOCK);
        __syncthreads();   // the list is rewritten by the next tile / slot
        tb0 = t1;
    }
}

// CTA-wide Random_N with many draws: draw -> rank sort into list.  Contains barriers.
template <int NT>
__device__ __noinline__ void random_n_sorted(const ItemCtx& cx, const VarDesc& vd, uint32_t* tmp, uint32_t* list) {
    const int n_bp = vd.n_bp;
    for (int call = threadIdx.x; call * 4 < n_bp; call += NT) {
        const U4 r = random_n_words(cx.seed, cx.seq_id, (uint32_t)vd.rng_id, (uint32_t)call);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) if (call * 4 + t < n_bp) tmp[call * 4 + t] = random_n_entry(w[t], cx.L);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_bp; i += NT) {
        const uint32_t e = tmp[i];
        int rank = 0;
        for (int j = 0; j < n_bp; ++j) { const uint32_t ej = tmp[j]; rank += (ej < e || (ej == e && j < i)) ? 1 : 0; }
        list[rank] = e;
    }
    __syncthreads();
}
template <int K, int NT>
__device__ __forceinline__ void random_n_list(ProfSmem<K, NT>& sm, const ItemCtx& cx, const VarDesc& vd, uint32_t* tmp) {
    random_n_sorted<NT>(cx, vd, tmp, sm.list);
}

// LONG path (L > 65535): patch hist[] itself (int32 counts), one variant at a time.
template <int K, int NT, int OUT>
__device__ __noinline__ void long_path(ProfSmem<K, NT>& sm, const ProfParams& p, const ItemCtx& cx, const VarDesc* vars,
                                       const long long* out_offs, long long item, long long seq, int base_total) {
    using C = ProfCfg<K, NT>;
    constexpr int VEC = C::VEC, VPT = C::VPT;
    constexpr int ESZ = (OUT == IDL_OUT_FREQ_F64 || OUT == IDL_OUT_CANON_F64) ? 8 : 4;
    const int tid = threadIdx.x, lane = tid & 31;
    const int L = cx.L;
    const int nblocks = (L + RNG_BLOCK - 1) / RNG_BLOCK;
    for (int s = 0; s < p.S; ++s) {
        const VarDesc vd = vars[p.sel ? p.sel[item * p.S + s] : s];
        const int kind = (vd.kind == KIND_RANDOM_N && vd.n_bp <= 0) ? KIND_CLEAN : vd.kind;
        if (tid == 0) sm.dtot[0] = 0;
        __syncthreads();
        int n_list = 0;
        const uint32_t* lst = sm.list;
        if (kind == KIND_RANDOM_N) {
            random_n_list<K, NT>(sm, cx, vd, sm.privtmp);
            n_list = vd.n_bp;
        } else if (kind == KIND_EXPLICIT) {
            const long long li = (long long)vd.explicit_idx * p.n_seqs_total + seq;
            lst = p.edits + p.edit_off[li];
            n_list = (int)(p.edit_off[li + 1] - p.edit_off[li]);
        }
        for (int sgn = 1; sgn >= -1; sgn -= 2) {
            if (kind == KIND_CLEAN) { if (sgn < 0) break; }
            else if (kind == KIND_RANDOM_N || kind == KIND_EXPLICIT) {
                int d = 0;
                for (int i = tid; i < n_list; i += NT) d += apply_hist<K>(cx, lst, n_list, i, sm.hist, sgn);
                if (sgn > 0) { d = warp_sum(d); if (lane == 0 && d) atomicAdd(&sm.dtot[0], d); }
                __syncthreads();
            } else {
                bern_tiles<K, NT>(sm, p, cx, vd, nblocks, [&](int total, int lo, long long hi) {
                    int d = 0;
                    for (int i = tid; i < total; i += NT) {
                        const int pos = (int)(sm.list[i] >> 3);
                        if (pos >= lo && pos < hi) d += apply_hist<K>(cx, sm.list, total, i, sm.hist, sgn);
                    }
                    if (sgn > 0) { d = warp_sum(d); if (lane == 0 && d) atomicAdd(&sm.dtot[0], d); }
                });
            }
            if (sgn > 0) {
                const int total = base_total + sm.dtot[0];
                const float ftot = (float)total;
                const float y = 1.0f / ftot;
                const bool big = total >= (1 << 24);
                void* row = reinterpret_cast<unsigned char*>(p.out) + (size_t)ESZ * (size_t)(out_offs[s] + item * p.out_stride);
                if constexpr (is_canon(OUT)) {
                    emit_canon_row<K, NT, OUT>(row, [&](uint32_t m) { return sm.hist[m] + p.pseudocount; }, p.mean, p.scale, sm.scan);
                } else {
#pragma unroll
                for (int vv = 0; vv < VPT; ++vv) {
                    const int vec = tid + vv * NT;
                    if (VEC % NT != 0 && vec >= VEC) break;
                    const int4 h = reinterpret_cast<const int4*>(sm.hist)[vec];
                    const int ci[4] = {h.x + p.pseudocount, h.y + p.pseudocount, h.z + p.pseudocount, h.w + p.pseudocount};
                    const float cf[4] = {(float)ci[0], (float)ci[1], (float)ci[2], (float)ci[3]};
                    float mean[4] = {0.f, 0.f, 0.f, 0.f}, scale[4] = {1.f, 1.f, 1.f, 1.f}, rscale[4] = {1.f, 1.f, 1.f, 1.f};
                    if (OUT == IDL_OUT_STD_F32) {
                        const float4 m = reinterpret_cast<const float4*>(p.mean)[vec];
                        const float4 sc = reinterpret_cast<const float4*>(p.scale)[vec];
                        mean[0] = m.x; mean[1] = m.y; mean[2] = m.z; mean[3] = m.w;
                        const float4 rs = reinterpret_cast<const float4*>(p.rscale)[vec];
                        scale[0] = sc.x; scale[1] = sc.y; scale[2] = sc.z; scale[3] = sc.w;
                        rscale[0] = rs.x; rscale[1] = rs.y; rscale[2] = rs.z; rscale[3] = rs.w;
                    }
                    emit_granule<OUT>(row, vec, ci, cf, total, ftot, y, big, p.accumulate, mean, scale, rscale);
                }
                }
                __syncthreads();
            }
        }
    }
}

// CTA-wide prep of the Bernoulli / explicit / big-Random_N slots of one group (short path):
// patches the private copies and accumulates sm.dtot.  Contains barriers (uniform control flow).
template <int K, int NT>
__device__ __noinline__ void prep_cta_slots(ProfSmem<K, NT>& sm, const ProfParams& p, const ItemCtx& cx, const VarDesc* vars, int s0,
                                            long long item, long long seq, unsigned bern_mask, unsigned other_mask, int* dtot, int copy0) {
    using C = ProfCfg<K, NT>;
    constexpr int PRIVW = C::PRIVW;
    const int tid = threadIdx.x, lane = tid & 31;
    const int L = cx.L;
    const int nblocks = (L + RNG_BLOCK - 1) / RNG_BLOCK;
    uint32_t* priv = sm.privtmp + copy0 * PRIVW;
    auto slot_var = [&](int slot) -> int { return p.sel ? p.sel[item * p.S + slot] : slot; };
    // ---- Bernoulli slots jointly: thread <-> (slot, 64-base block), mask generator ----
    const int nb = __popc(bern_mask);
    bool bern_done = nb == 0;
    if (nb > 0 && nb * nblocks <= NT) {
        const int j = tid / nblocks, b = tid - j * nblocks;
        const bool active = tid < nb * nblocks;
        const int c = active ? (int)__fns(bern_mask, 0, j + 1) : 0;
        const VarDesc vd = vars[slot_var(s0 + c)];
        BlockMasks m;
        m.a = m.b = m.ch = 0;
        if (active)
            m = block_masks(vd.kind, cx.seed, cx.seq_id, (uint32_t)vd.rng_id, b, L, cx.nmask, gap_table(sm, p, vd.tab1), vd.slope1,
                            gap_table(sm, p, vd.tab2), vd.slope2);
        int total;
        const int off = block_exscan<NT>(block_masks_count(m), sm.scan, &total);
        if (total <= LIST_CAP) {  // uniform
            bern_done = true;
            if (active && b == 0) sm.seg_off[j] = off;
            if (tid == 0) sm.seg_off[nb] = total;
            block_masks_write(m, b, cx.codes, sm.list + off);
            __syncthreads();
            for (int i = tid; i < total; i += NT) {
                int jj = 0;
                while (i >= sm.seg_off[jj + 1]) ++jj;
                const int cc = (int)__fns(bern_mask, 0, jj + 1);
                const int so = sm.seg_off[jj];
                const int d = apply_priv<K>(cx, sm.list + so, sm.seg_off[jj + 1] - so, i - so, priv + cc * PRIVW);
                if (d) atomicAdd(&dtot[cc], d);
            }
            __syncthreads();
        }
    }
    // ---- remaining CTA-wide slots, one after the other ----
    unsigned todo = other_mask | (bern_done ? 0u : bern_mask);
    while (todo) {
        const int c = __ffs(todo) - 1;
        todo &= todo - 1;
        const VarDesc vd = vars[slot_var(s0 + c)];
        uint32_t* privc = priv + c * PRIVW;
        int d = 0;
        if (vd.kind == KIND_EXPLICIT) {
            const long long li = (long long)vd.explicit_idx * p.n_seqs_total + seq;
            const uint32_t* glist = p.edits + p.edit_off[li];
            const int n = (int)(p.edit_off[li + 1] - p.edit_off[li]);
            for (int i = tid; i < n; i += NT) d += apply_priv<K>(cx, glist, n, i, privc);
        } else if (vd.kind == KIND_RANDOM_N) {
            random_n_list<K, NT>(sm, cx, vd, sm.list + LIST_CAP / 2);
            for (int i = tid; i < vd.n_bp; i += NT) d += apply_priv<K>(cx, sm.list, vd.n_bp, i, privc);
        } else {
            bern_tiles<K, NT>(sm, p, cx, vd, nblocks, [&](int total, int lo, long long hi) {
                for (int i = tid; i < total; i += NT) {
                    const int pos = (int)(sm.list[i] >> 3);
                    if (pos >= lo && pos < hi) d += apply_priv<K>(cx, sm.list, total, i, privc);
                }
            });
        }
        d = warp_sum(d);
        if (lane == 0 && d) atomicAdd(&dtot[c], d);
        __syncthreads();
    }
}

template <int K, int NT, int OUT>
__global__ void __launch_bounds__(NT, (K == 6 ? 2 : K == 5 ? 4 : 8)) profiles_kernel(const ProfParams p, const __grid_constant__ Plan plan) {
    using C = ProfCfg<K, NT>;
    constexpr int F = C::F, VEC = C::VEC, VPT = C::VPT, G = C::G, PRIVW = C::PRIVW;
    constexpr int ESZ = (OUT == IDL_OUT_FREQ_F64 || OUT == IDL_OUT_CANON_F64) ? 8 : 4;
    constexpr bool NEED_F = (OUT == IDL_OUT_FREQ_F32 || OUT == IDL_OUT_STD_F32);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ProfSmem<K, NT>& sm = *reinterpret_cast<ProfSmem<K, NT>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (p.only_deferred && p.work_counter[1] == 0ull) {   // the fast kernel took every item (stream order: its count is final)
        if (OUT == OUT_STATS && tid == 0) p.stats_n[blockIdx.x] = 0.0;   // an empty part
        return;
    }

    const float magic = 8388608.0f - (float)p.pseudocount;
    const bool cached = p.inline_plan != 0;
    if (cached) {
        for (int i = tid; i < p.n_vars; i += NT) sm.svars[i] = plan.vars[i];
        for (int i = tid; i < p.S; i += NT) sm.sout_off[i] = plan.out_off[i];
    }
    for (int i = tid; i < STABS * RNG_BLOCK; i += NT)
        (&sm.gtabs[0][0])[i] = i < p.n_tabs * RNG_BLOCK ? (cached ? (&plan.gtab[0][0])[i] : p.gtab[i]) : 0u;
    const VarDesc* __restrict__ vars = cached ? sm.svars : p.vars;
    const long long* __restrict__ out_offs = cached ? sm.sout_off : reinterpret_cast<const long long*>(p.out_off);

    // OUT_STATS: shifted-data column sums of this CTA's rows (shift = first row seen), float64
    double acc1[VPT][4], acc2[VPT][4];
    float shiftK[VPT][4];
    int n_acc = 0;
    long long stats_cursor = blockIdx.x;   // OUT_STATS: next own item (thread 0; every thread in deferred mode)
    long long dq_base = 0;                 // deferred mode: first item of the NT examined last
    int dq_pos = NT;                       // deferred mode: next bit of sm.dqmask to look at (NT: refill)
#pragma unroll
    for (int vv = 0; vv < VPT; ++vv)
#pragma unroll
        for (int e = 0; e < 4; ++e) { acc1[vv][e] = 0.0; acc2[vv][e] = 0.0; shiftK[vv][e] = 0.f; }
    for (;;) {
        __syncthreads();  // previous item fully done (also protects sm.item)
        long long item;
        if (p.only_deferred) {
            // deferred mode: the CTA looks at NT status words at a time (one per thread, ballot masks in shared memory)
            // instead of one global round trip per item examined.  OUT_STATS: static rows per CTA (its own items in
            // ascending order -> reproducible sums); otherwise chunks of NT items from a global cursor.
            for (;;) {
                item = -1;
                while (dq_pos < NT) {
                    const unsigned w = sm.dqmask[dq_pos >> 5] >> (dq_pos & 31);
                    if (w) {
                        const int b = dq_pos + __ffs(w) - 1;
                        dq_pos = b + 1;
                        item = dq_base + (OUT == OUT_STATS ? (long long)b * gridDim.x : (long long)b);
                        break;
                    }
                    dq_pos = (dq_pos | 31) + 1;
                }
                if (item >= 0) break;
                __syncthreads();   // everybody is done with the old masks
                if (OUT == OUT_STATS) { dq_base = stats_cursor; stats_cursor += (long long)NT * gridDim.x; }
                else {
                    if (tid == 0) sm.item = (long long)atomicAdd(p.work_counter + 2, (unsigned long long)NT);
                    __syncthreads();
                    dq_base = sm.item;
                }
                if (dq_base >= p.n_items) { item = p.n_items; break; }
                const long long it = dq_base + (OUT == OUT_STATS ? (long long)tid * gridDim.x : (long long)tid);
                const bool hit = it < p.n_items && (p.status[it] & 2);
                if (hit) atomicAnd(p.status + it, ~2);
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                if (lane == 0) sm.dqmask[wid] = m;
                __syncthreads();
                dq_pos = 0;
            }
        } else {
            if (tid == 0) {
                long long it;
                if (OUT == OUT_STATS) { it = stats_cursor; stats_cursor = it + gridDim.x; }   // static rows per CTA: reproducible sums
                else it = (long long)atomicAdd(p.work_counter, 1ull);
                sm.item = it;
            }
            __syncthreads();
            item = sm.item;
        }
        if (item >= p.n_items) break;
        const long long seq = p.sidx ? (long long)p.sidx[item] : item;
        ItemCtx cx;
        cx.L = p.len[seq];
        const long long c0 = p.chunk_off[seq];
        cx.codes = p.codes + c0 * 4;
        cx.nmask = p.nmask + c0 * 2;
        cx.seq_id = (uint32_t)(p.seq_id0 + seq);
        cx.seed = p.seed;
        const int L = cx.L;
        if (p.long_overflow && L >= CH_MIN_LEN && *p.long_overflow == 0) continue;   // the chunked path owns the item
        const int nhalf = ((L + CHUNK_BASES - 1) / CHUNK_BASES) * 2;
        const bool staged = nhalf <= 2 * SSEQ_CHUNKS;
        auto slot_var = [&](int slot) -> int { return p.sel ? p.sel[item * p.S + slot] : slot; };

        // ---- clean histogram -------------------------------------------------------------
        for (int i = tid; i < VEC; i += NT) reinterpret_cast<int4*>(sm.hist)[i] = make_int4(0, 0, 0, 0);
        if (tid == 0) sm.nvalid = 0;
        __syncthreads();
        {
            int nv = 0;
            for (int h = tid; h < nhalf; h += NT) {
                const uint2 w = __ldg(reinterpret_cast<const uint2*>(cx.codes) + h);
                if (staged) {
                    reinterpret_cast<uint2*>(sm.sseq)[h] = w;
                    sm.sseq[SSEQ_CW + h] = cx.nmask[h];
                }
                nv += count_half<K>(cx.codes, cx.nmask, h, w.x, w.y, [&](uint32_t kmer) { atomicAdd(&sm.hist[kmer], 1); });
            }
            if (staged) {  // slack chunk behind the sequence (window reads run one word past the end)
                if (tid < 4) sm.sseq[nhalf * 2 + tid] = 0u;
                if (tid < 2) sm.sseq[SSEQ_CW + nhalf + tid] = 0xFFFFFFFFu;
            }
            nv = warp_sum(nv);
            if (lane == 0 && nv) atomicAdd(&sm.nvalid, nv);
        }
        __syncthreads();
        const int base_total = F * p.pseudocount + sm.nvalid;
        if (staged) { cx.codes = sm.sseq; cx.nmask = sm.sseq + SSEQ_CW; }  // every later lookup hits shared memory

        if (OUT == OUT_STATS) {
            // ---- statistics mode: patch hist[] in place with slot 0's deltas, accumulate, next item ----
            const VarDesc vd = vars[slot_var(0)];
            if (tid == 0) sm.dtot[0] = 0;
            __syncthreads();
            const int nblk = (L + RNG_BLOCK - 1) / RNG_BLOCK;
            const bool bern = vd.kind == KIND_TRANSITION || vd.kind == KIND_TRANSVERSION || vd.kind == KIND_BOTH;
            if (bern && nblk > 0) {
                bern_tiles<K, NT>(sm, p, cx, vd, nblk, [&](int total, int lo, long long hi) {
                    int d = 0;
                    for (int i = tid; i < total; i += NT) {
                        const int pos = (int)(sm.list[i] >> 3);
                        if (pos >= lo && pos < hi) d += apply_hist<K>(cx, sm.list, total, i, sm.hist, 1);
                    }
                    d = warp_sum(d);
                    if (lane == 0 && d) atomicAdd(&sm.dtot[0], d);
                });
            }
            if (vd.kind == KIND_EXPLICIT || (vd.kind == KIND_RANDOM_N && vd.n_bp > 0 && L > 0)) {
                const uint32_t* lst = sm.list;
                int n_list = vd.n_bp;
                if (vd.kind == KIND_EXPLICIT) {
                    const long long li = (long long)vd.explicit_idx * p.n_seqs_total + seq;
                    lst = p.edits + p.edit_off[li];
                    n_list = (int)(p.edit_off[li + 1] - p.edit_off[li]);
                } else {
                    random_n_list<K, NT>(sm, cx, vd, sm.privtmp);
                }
                int d = 0;
                for (int i = tid; i < n_list; i += NT) d += apply_hist<K>(cx, lst, n_list, i, sm.hist, 1);
                d = warp_sum(d);
                if (lane == 0 && d) atomicAdd(&sm.dtot[0], d);
            }
            __syncthreads();
            const int total = base_total + sm.dtot[0];
            const float ftot = (float)total;
            const float y = 1.0f / ftot;
            const bool big = total >= (1 << 24);
#pragma unroll
            for (int vv = 0; vv < VPT; ++vv) {
                const int vec = tid + vv * NT;
                if (VEC % NT != 0 && vec >= VEC) break;
                const int4 h = reinterpret_cast<const int4*>(sm.hist)[vec];
                const int ci[4] = {h.x + p.pseudocount, h.y + p.pseudocount, h.z + p.pseudocount, h.w + p.pseudocount};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float q = big ? (float)((double)ci[e] / (double)total) : div_rn((float)ci[e], ftot, y);
                    if (n_acc == 0) shiftK[vv][e] = q;
                    const double dd = (double)q - (double)shiftK[vv][e];
                    acc1[vv][e] += dd;
                    acc2[vv][e] = fma(dd, dd, acc2[vv][e]);
                }
            }
            ++n_acc;
            continue;
        }
        if (L > 65535) {
            long_path<K, NT, OUT>(sm, p, cx, vars, out_offs, item, seq, base_total);
            continue;
        }
        // =================================== SHORT path ===================================
        uint32_t* priv = sm.privtmp;
        // pack the clean histogram to uint16: G private copies + one pristine copy that overwrites
        // (the first half of) the int32 histogram in place and restores the copies while streaming
        uint2* clean16 = reinterpret_cast<uint2*>(sm.hist);
        {
            uint2 pk[VPT];
#pragma unroll
            for (int vv = 0; vv < VPT; ++vv) {
                const int vec = tid + vv * NT;
                pk[vv] = make_uint2(0u, 0u);
                if (VEC % NT == 0 || vec < VEC) {
                    const int4 h = reinterpret_cast<const int4*>(sm.hist)[vec];
                    pk[vv] = make_uint2((uint32_t)h.x | ((uint32_t)h.y << 16), (uint32_t)h.z | ((uint32_t)h.w << 16));
                }
            }
            __syncthreads();  // every int32 bin has been read before the region is overwritten
#pragma unroll
            for (int vv = 0; vv < VPT; ++vv) {
                const int vec = tid + vv * NT;
                if (VEC % NT == 0 || vec < VEC) {
                    clean16[vec] = pk[vv];
#pragma unroll
                    for (int c = 0; c < G; ++c) reinterpret_cast<uint2*>(priv + c * PRIVW)[vec] = pk[vv];
                }
            }
        }

        for (int S0 = 0; S0 < p.S;) {
            // ======== supergroup: up to SG slots; their Random_N removals are precomputed together ========
            __syncthreads();  // copies initialised / restored; previous supergroup's tables no longer read
            if (wid == 0) {
                const int ns_try = p.S - S0 < SG ? p.S - S0 : SG;
                int kc = 0, nb = 0;
                if (lane < ns_try) {
                    const VarDesc vd = vars[slot_var(S0 + lane)];
                    if (vd.kind == KIND_RANDOM_N) kc = (L == 0 || vd.n_bp <= 0) ? 0 : (vd.n_bp <= 32 ? 1 : 3);
                    else if (vd.kind == KIND_EXPLICIT) kc = 3;
                    else if (vd.kind != KIND_CLEAN) kc = L > 0 ? 2 : 0;
                    nb = kc == 1 ? vd.n_bp : 0;
                }
                int inc = nb;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                const bool fits = inc * K <= REM_CAP && inc <= ENT_CAP;
                const unsigned fm = __ballot_sync(0xffffffffu, fits);
                int nfit = fm == 0xffffffffu ? 32 : __ffs(~fm) - 1;
                int nsg = ns_try < nfit ? ns_try : nfit;
                if (nsg < ns_try) nsg = (nsg / G) * G;   // a whole number of groups (one group always fits)
                if (lane < nsg) {
                    sm.pre_kind[lane] = kc; sm.pre_off[lane] = inc - nb; sm.pre_nbp[lane] = nb;
                    sm.dtot[lane] = 0;
                    sm.grow[lane] = (long long)ESZ * (out_offs[S0 + lane] + item * p.out_stride);
                }
                const unsigned mb = __ballot_sync(0xffffffffu, lane < nsg && kc == 2);
                const unsigned mo = __ballot_sync(0xffffffffu, lane < nsg && kc == 3);
                const int ent_total = __shfl_sync(0xffffffffu, inc, nsg > 0 ? nsg - 1 : 0);
                if (lane == 0) { sm.sg_n = nsg; sm.sg_ent = nsg > 0 ? ent_total : 0; sm.mask_bern = mb; sm.mask_other = mo; }
            }
            __syncthreads();
            const int NSg = sm.sg_n;
            // ---- (p1) draws of every small Random_N slot: thread <-> (slot, philox call).  The slot id
            // ---- rides in bits 27..31 of the entry (positions are < 2^16 on this path) ----
            for (int q = tid; q < NSg * 8; q += NT) {
                const int c = q >> 3, j = q & 7;
                const int nb = sm.pre_nbp[c];
                if (4 * j < nb) {
                    const U4 r = random_n_words(p.seed, cx.seq_id, (uint32_t)vars[slot_var(S0 + c)].rng_id, (uint32_t)j);
                    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
                    uint32_t* dst = sm.list + sm.pre_off[c] + 4 * j;
#pragma unroll
                    for (int t = 0; t < 4; ++t) if (4 * j + t < nb) dst[t] = random_n_entry(w[t], L) | ((uint32_t)c << 27);
                }
            }
            __syncthreads();
            // ---- (p2) removed windows of every draw: thread <-> draw (dense over all slots); draw q
            // ---- owns rem[q*K .. +K), unused entries hold 0xFFFF (random_n_removals' rule, core.cuh) ----
            {
                constexpr uint32_t KMASK = (1u << (2 * K)) - 1u, NMASKK = (1u << K) - 1u;
                const int n_ent = sm.sg_ent;
                for (int q = tid; q < n_ent; q += NT) {
                    const uint32_t me = sm.list[q];
                    const int c = (int)(me >> 27);
                    const int nb = sm.pre_nbp[c], off = sm.pre_off[c], i = q - off;
                    const uint32_t pme = me >> 3;            // position | slot bits: comparable within the slot
                    uint32_t pnx = 0xFFFFFFFFu;
                    bool dup = false;
                    const uint32_t* e = sm.list + off;
                    int j = 0;
                    if ((off & 3) == 0) {
                        for (; j + 4 <= nb; j += 4) {
                            const uint4 v = *reinterpret_cast<const uint4*>(e + j);
                            const uint32_t pv[4] = {v.x >> 3, v.y >> 3, v.z >> 3, v.w >> 3};
#pragma unroll
                            for (int t = 0; t < 4; ++t) {
                                dup = dup || (pv[t] == pme && j + t < i);
                                if (pv[t] > pme && pv[t] < pnx) pnx = pv[t];
                            }
                        }
                    }
                    for (; j < nb; ++j) {
                        const uint32_t pj = e[j] >> 3;
                        dup = dup || (pj == pme && j < i);
                        if (pj > pme && pj < pnx) pnx = pj;
                    }
                    uint16_t* dst = sm.rem + q * K;
                    int cnt = 0;
                    if (!dup) {
                        const int pos = (int)(pme & 0xFFFFFFu);
                        int e_hi = pos + K - 1;
                        if (pnx != 0xFFFFFFFFu && (int)(pnx & 0xFFFFFFu) - 1 < e_hi) e_hi = (int)(pnx & 0xFFFFFFu) - 1;
                        if (L - 1 < e_hi) e_hi = L - 1;
                        const Window<K> cw = load_window<K>(cx.codes, cx.nmask, pos - (K - 1));
                        for (int ee = pos; ee <= e_hi; ++ee) {
                            const int sh = K - 1 - (ee - pos);
                            if (((cw.nbits >> sh) & NMASKK) == 0u) dst[cnt++] = (uint16_t)((cw.bases >> (2 * sh)) & KMASK);
                        }
                    }
                    for (int r = cnt; r < K; ++r) dst[r] = 0xFFFFu;
                }
            }
            __syncthreads();
            for (int c = wid; c < NSg; c += NT / 32) {  // totals of the slots whose deltas are known now: warp <-> slot
                int d = 0;
                if (sm.pre_kind[c] == 1) {
                    const uint16_t* rl = sm.rem + sm.pre_off[c] * K;
                    const int n = sm.pre_nbp[c] * K;
                    for (int r = lane; r < n; r += 32) d -= rl[r] != 0xFFFFu ? 1 : 0;
                    d = warp_sum(d);
                }
                if (lane == 0) {
                    if (sm.pre_kind[c] == 1) sm.dtot[c] = d;
                    const float ft2 = (float)(base_total + d);
                    sm.gy[c] = make_float2(ft2, 1.0f / ft2);
                }
            }
            // (visible to the streamers after the barrier that follows the first patch phase)

            // ---- half-groups of HG slots, two sets of private copies: the removals of the NEXT
            // ---- half-group are subtracted (fire-and-forget shared atomics) while the current one streams
            constexpr int HG = G / 2 > 0 ? G / 2 : 1;
            constexpr int TPH = NT / HG;
            const unsigned cta_mask = sm.mask_bern | sm.mask_other;
            auto patch_half = [&](int h0, int hs, int set) {
                const int c = tid / TPH;
                if (c < hs && sm.pre_kind[h0 + c] == 1) {
                    const int n = sm.pre_nbp[h0 + c] * K;
                    const uint16_t* rl = sm.rem + sm.pre_off[h0 + c] * K;
                    uint32_t* privc = priv + (set * HG + c) * PRIVW;
                    for (int r = tid - c * TPH; r < n; r += TPH) {
                        const uint32_t km = rl[r];
                        if (km != 0xFFFFu) upd16(privc, km, -1);
                    }
                }
            };
            auto prep_half = [&](int h0, int hs, int set) {  // CTA-wide slots of a half-group (contains barriers)
                const unsigned bm = (sm.mask_bern >> h0) & ((1u << HG) - 1u), om = (sm.mask_other >> h0) & ((1u << HG) - 1u);
                prep_cta_slots<K, NT>(sm, p, cx, vars, S0 + h0, item, seq, bm, om, sm.dtot + h0, set * HG);
                if (tid < hs && sm.pre_kind[h0 + tid] >= 2) {
                    const float ft2 = (float)(base_total + sm.dtot[h0 + tid]);
                    sm.gy[h0 + tid] = make_float2(ft2, 1.0f / ft2);
                }
            };
            const int nh = (NSg + HG - 1) / HG;
            if ((cta_mask & ((1u << HG) - 1u)) != 0u) { __syncthreads(); prep_half(0, NSg < HG ? NSg : HG, 0); }
            patch_half(0, NSg < HG ? NSg : HG, 0);
            __syncthreads();
            for (int h = 0; h < nh; ++h) {
                const int cur = h & 1, h0 = h * HG;
                const int hs = NSg - h0 < HG ? NSg - h0 : HG;
                const bool has_next = h + 1 < nh;
                const int hs_next = has_next ? (NSg - h0 - HG < HG ? NSg - h0 - HG : HG) : 0;
                const bool next_cta = has_next && ((cta_mask >> (h0 + HG)) & ((1u << HG) - 1u)) != 0u;
                if (has_next && !next_cta) patch_half(h0 + HG, hs_next, cur ^ 1);
                if constexpr (is_canon(OUT)) {
                    // ---- canonical rows read both bins of a reverse-complement pair, which other threads' granules hold:
                    // ---- slot by slot from the copies, then (after every read) the copies are restored ----
                    for (int c = 0; c < hs; ++c) {
                        const uint32_t* cp = priv + (cur * HG + c) * PRIVW;
                        emit_canon_row<K, NT, OUT>(
                            reinterpret_cast<unsigned char*>(p.out) + sm.grow[h0 + c],
                            [&](uint32_t m) { return (int)((cp[m >> 1] >> ((m & 1u) * 16u)) & 0xFFFFu) + p.pseudocount; }, p.mean, p.scale, sm.scan);
                    }
                    __syncthreads();
#pragma unroll
                    for (int vv = 0; vv < VPT; ++vv) {
                        const int vec = tid + vv * NT;
                        if (VEC % NT != 0 && vec >= VEC) break;
                        const uint2 clean = clean16[vec];
                        for (int c = 0; c < hs; ++c) reinterpret_cast<uint2*>(priv + (cur * HG + c) * PRIVW)[vec] = clean;
                    }
                } else {
                // ---- stream the hs profiles of this half-group (and restore its copies) ----
                // granule-major: the scaler statistics of ONE granule (12 registers) are live at a time
#pragma unroll
                for (int vv = 0; vv < VPT; ++vv) {
                    const int vec = tid + vv * NT;
                    if (VEC % NT != 0 && vec >= VEC) break;
                    const Stats2 st2 = load_stats2(p.mean, p.scale, p.rscale, vec, OUT == IDL_OUT_STD_F32);
                    const float mean[4] = {0.f, 0.f, 0.f, 0.f}, scale[4] = {1.f, 1.f, 1.f, 1.f}, rscale[4] = {1.f, 1.f, 1.f, 1.f};
                    const uint2 clean = clean16[vec];
#pragma unroll 2
                    for (int c = 0; c < hs; ++c) {
                        const float2 fy = sm.gy[h0 + c];
                        unsigned char* row = reinterpret_cast<unsigned char*>(p.out) + sm.grow[h0 + c];
                        uint2* src = reinterpret_cast<uint2*>(priv + (cur * HG + c) * PRIVW);
                        const uint2 pk = src[vec];
                        src[vec] = clean;  // the copy is clean again for its next user
                        if (NEED_F) {
                            emit_granule_u16x2<OUT == IDL_OUT_STD_F32>(row, vec, pk, magic, fy, st2);
                        } else {
                            int ci[4];
                            const float cf[4] = {0.f, 0.f, 0.f, 0.f};
                            ci[0] = (int)(pk.x & 0xFFFFu) + p.pseudocount; ci[1] = (int)(pk.x >> 16) + p.pseudocount;
                            ci[2] = (int)(pk.y & 0xFFFFu) + p.pseudocount; ci[3] = (int)(pk.y >> 16) + p.pseudocount;
                            emit_granule<OUT>(row, vec, ci, cf, base_total + sm.dtot[h0 + c], fy.x, fy.y, false, p.accumulate, mean, scale, rscale);
                        }
                    }
                }
                }
                __syncthreads();
                if (next_cta) {
                    prep_half(h0 + HG, hs_next, cur ^ 1);
                    patch_half(h0 + HG, hs_next, cur ^ 1);
                    __syncthreads();
                }
            }
            S0 += NSg;
        }
    }
    if (OUT == OUT_STATS) {   // this CTA's part: (rows, mean, M2) per column, merged by scaler_finalize_kernel
        if (tid == 0) p.stats_n[blockIdx.x] = (double)n_acc;
        const double m = n_acc > 0 ? (double)n_acc : 1.0;
#pragma unroll
        for (int vv = 0; vv < VPT; ++vv) {
            const int vec = tid + vv * NT;
            if (VEC % NT != 0 && vec >= VEC) break;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                p.stats_partials[((size_t)blockIdx.x * 2 + 0) * F + vec * 4 + e] = (double)shiftK[vv][e] + acc1[vv][e] / m;
                p.stats_partials[((size_t)blockIdx.x * 2 + 1) * F + vec * 4 + e] = acc2[vv][e] - acc1[vv][e] * acc1[vv][e] / m;
            }
        }
    }
}

}  // namespace idl
#include "profiles_pc.cuh"
#include "prep.cuh"
#include "chunked.cuh"
namespace idl {

// ---------------------------------------------------------------------------------------
// K4: column statistics / scaler / standardise
// ---------------------------------------------------------------------------------------
constexpr int CS_NT = 128;
// rows per partial: 256 for small matrices (enough CTAs to fill the GPU), more when that would mean over 1024 parts
static inline long long cs_rows(long long n) { const long long r = (n + 1023) / 1024; return r > 256 ? r : 256; }

template <typename T>
__global__ void __launch_bounds__(CS_NT) colstats_kernel(const T* __restrict__ x, long long n, int F, long long rows_per_part,
                                                          double* __restrict__ partials, double* __restrict__ part_n) {
    const int col = blockIdx.x * CS_NT + threadIdx.x;
    const long long r0 = (long long)blockIdx.y * rows_per_part;
    const long long r1 = r0 + rows_per_part < n ? r0 + rows_per_part : n;
    if (col == 0) part_n[blockIdx.y] = (double)(r1 - r0);
    if (col >= F) return;
    // shifted-data sums (shift = first row of this part): exact zeros for a constant column
    const double shift = (double)x[r0 * F + col];
    double s1 = 0.0, s2 = 0.0;
    for (long long r = r0; r < r1; ++r) {
        const double d = (double)x[r * F + col] - shift;
        s1 += d;
        s2 = fma(d, d, s2);
    }
    const double m = (double)(r1 - r0);
    partials[((long long)blockIdx.y * 2 + 0) * F + col] = shift + s1 / m;  // mean of the part
    partials[((long long)blockIdx.y * 2 + 1) * F + col] = s2 - s1 * s1 / m;  // M2 of the part
}

// Merge of the (rows, mean, M2) parts in index order (Chan et al.), one lane per column.  The chain over the parts is
// sequential per column and only 4^k columns exist, so a thread-per-column loop is bound by the latency of its own loads
// (0.10 ms for 592 parts at k = 6).  Here a CTA owns SF_COLS columns: all its threads fetch the next SF_PCH parts' rows (empty
// parts are skipped) while warp 0 runs the recurrence on the current ones out of shared memory; the weights nb / (na + nb) and
// na * nb / (na + nb) depend on the row counts alone and are computed once per part.  Same operations in the same order per
// column as the plain loop (bit-identical results).
constexpr int SF_COLS = 32, SF_NT = 256, SF_PCH = 64;
constexpr int SF_LD = SF_PCH * SF_COLS * 2 / 2 / SF_NT;   // double2 loads per thread and chunk
__global__ void __launch_bounds__(SF_NT) scaler_finalize_kernel(const double* __restrict__ partials, const double* __restrict__ part_n, int n_parts,
                                                                int F, double* mean64, double* var64, double* scale64, float* mean32, float* scale32) {
    __shared__ __align__(16) double s_row[SF_PCH][2][SF_COLS];   // [part][mean | M2][column]
    __shared__ double s_nb[SF_PCH], s_w1[SF_PCH], s_w2[SF_PCH];
    const int tid = threadIdx.x, lane = tid & 31;
    const int col0 = blockIdx.x * SF_COLS;
    const bool vec_ok = (F % 2 == 0) && (col0 + SF_COLS <= F);
    double2 pre[SF_LD];
    auto fetch = [&](int g0) {   // rows of parts g0 .. g0 + SF_PCH - 1 -> registers (empty parts and the range past the end: not loaded)
#pragma unroll
        for (int r = 0; r < SF_LD; ++r) {
            const int unit = r * SF_NT + tid;
            const int part = unit / SF_COLS, w = unit % SF_COLS;   // SF_COLS double2 units per part: SF_COLS / 2 of the mean row, SF_COLS / 2 of the M2 row
            const int which = w / (SF_COLS / 2), c = (w % (SF_COLS / 2)) * 2;
            const int g = g0 + part;
            pre[r] = make_double2(0.0, 0.0);
            if (g < n_parts && part_n[g] > 0.0) {
                const double* src = partials + ((long long)g * 2 + which) * F + col0 + c;
                if (vec_ok) pre[r] = *reinterpret_cast<const double2*>(src);
                else { if (col0 + c < F) pre[r].x = src[0]; if (col0 + c + 1 < F) pre[r].y = src[1]; }
            }
        }
    };
    double ma = 0.0, M2 = 0.0, na_carry = 0.0;
    fetch(0);
    for (int g0 = 0; g0 < n_parts; g0 += SF_PCH) {
        const int m = n_parts - g0 < SF_PCH ? n_parts - g0 : SF_PCH;
        __syncthreads();   // the previous chunk's chain is done
#pragma unroll
        for (int r = 0; r < SF_LD; ++r) {
            const int unit = r * SF_NT + tid;
            const int part = unit / SF_COLS, w = unit % SF_COLS;
            *reinterpret_cast<double2*>(&s_row[part][w / (SF_COLS / 2)][(w % (SF_COLS / 2)) * 2]) = pre[r];
        }
        if (tid < 32) {   // rows merged before each part: a scan of row counts (integers: exact in any order), then the weights
            const int i0 = 2 * lane, i1 = 2 * lane + 1;
            double v0 = i0 < m ? part_n[g0 + i0] : 0.0, v1 = i1 < m ? part_n[g0 + i1] : 0.0;
            v0 = v0 > 0.0 ? v0 : 0.0; v1 = v1 > 0.0 ? v1 : 0.0;
            const double sum2 = v0 + v1;
            double inc = sum2;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            const double na0 = na_carry + (inc - sum2), na1 = na0 + v0;
            s_nb[i0] = v0; s_nb[i1] = v1;
            { const double nt = na0 + v0; s_w1[i0] = v0 / nt; s_w2[i0] = na0 * v0 / nt; }
            { const double nt = na1 + v1; s_w1[i1] = v1 / nt; s_w2[i1] = na1 * v1 / nt; }
            na_carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        __syncthreads();
        if (g0 + SF_PCH < n_parts) fetch(g0 + SF_PCH);   // in flight during the chain below
        if (tid < 32) {
            for (int i = 0; i < m; ++i) {
                if (!(s_nb[i] > 0.0)) continue;
                const double mb = s_row[i][0][lane];
                const double Mb = s_row[i][1][lane];
                const double w1 = s_w1[i], w2 = s_w2[i];
                const double delta = mb - ma;
                ma = ma + delta * w1;
                M2 = M2 + Mb + delta * delta * w2;
            }
        }
    }
    const int col = col0 + lane;
    if (tid >= 32 || col >= F) return;
    const double na = na_carry;
    double var = na > 0.0 ? M2 / na : 0.0;
    if (var < 0.0) var = 0.0;
    // sklearn/preprocessing/_data.py::_is_constant_feature (float64 eps) -> scale 1
    const double eps = 2.220446049250313e-16;
    const double bound = na * eps * var + (na * ma * eps) * (na * ma * eps);
    double sc = sqrt(var);
    if (var <= bound) sc = 1.0;
    if (mean64) mean64[col] = ma;
    if (var64) var64[col] = var;
    if (scale64) scale64[col] = sc;
    if (mean32) mean32[col] = (float)ma;
    if (scale32) scale32[col] = (float)sc;
}

__global__ void standardize_f32_kernel(const float* __restrict__ x, float* __restrict__ out, long long n4, int F4,
                                       const float* __restrict__ mean, const float* __restrict__ scale) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int cstep = (int)(stride % F4);
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int c = (int)(i % F4);   // column granule, advanced incrementally (a 64-bit modulo per element costs more than the element)
    for (; i < n4; i += stride, c = c + cstep >= F4 ? c + cstep - F4 : c + cstep) {
        const float4 v = reinterpret_cast<const float4*>(x)[i];
        const float4 m = __ldg(reinterpret_cast<const float4*>(mean) + c);
        const float4 s = __ldg(reinterpret_cast<const float4*>(scale) + c);
        float4 o;
        o.x = (v.x - m.x) / s.x; o.y = (v.y - m.y) / s.y; o.z = (v.z - m.z) / s.z; o.w = (v.w - m.w) / s.w;
        reinterpret_cast<float4*>(out)[i] = o;
    }
}

// any F and alignment (the canonical k-mer widths R = 2 and 10 of k = 1, 2 are not multiples of 4): one element per step,
// the same (x - mean32) / scale32 as standardize_f32_kernel.  x may be out (in place).
__global__ void standardize_f32_elem_kernel(const float* x, float* out, long long total, int F, const float* __restrict__ mean,
                                            const float* __restrict__ scale) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int cstep = (int)(stride % F);
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int c = (int)(i % F);
    for (; i < total; i += stride, c = c + cstep >= F ? c + cstep - F : c + cstep) out[i] = (x[i] - mean[c]) / scale[c];
}

__global__ void standardize_f64_kernel(const double* __restrict__ x, double* __restrict__ out64, float* __restrict__ out32,
                                       long long total, int F, const double* __restrict__ mean, const double* __restrict__ scale) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int cstep = (int)(stride % F);
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int c = (int)(i % F);
    for (; i < total; i += stride, c = c + cstep >= F ? c + cstep - F : c + cstep) {
        const double o = (x[i] - mean[c]) / scale[c];
        if (out64) out64[i] = o;
        if (out32) out32[i] = (float)o;
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// per-device facts: SM count, and which kernels already carry their dynamic shared-memory opt-in ON THAT DEVICE
// (cudaFuncSetAttribute is per device; a process may drive several)
static std::mutex g_dev_mu;
static int g_sm_counts[64];
static std::vector<std::pair<int, const void*>> g_smem_done;

static int sm_count() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    std::lock_guard<std::mutex> lk(g_dev_mu);
    if (g_sm_counts[dev] == 0 && cudaDeviceGetAttribute(&g_sm_counts[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) g_sm_counts[dev] = 148;
    return g_sm_counts[dev];
}
static cudaError_t ensure_dyn_smem(const void* func, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_dev_mu);
    for (const auto& d : g_smem_done)
        if (d.first == dev && d.second == func) return cudaSuccess;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) g_smem_done.emplace_back(dev, func);
    return e;
}
// grid of a persistent kernel: as many CTAs as fit on every SM (at most cta_cap per SM when cta_cap > 0), at most one per item
template <typename Kernel>
static int persistent_grid(Kernel kern, int nt, size_t smem, int cta_cap, long long n_items, const char* name, unsigned& grid) {
    IDL_CUDA_CHECK(ensure_dyn_smem((const void*)kern, smem));
    int per_sm = 0;
    IDL_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nt, smem));
    if (per_sm < 1) return set_error(IDL_ECUDA, "%s kernel does not fit on an SM", name);
    if (cta_cap > 0 && per_sm > cta_cap) per_sm = cta_cap;   // the caller wants room left on every SM (a concurrent stream)
    const long long g = (long long)sm_count() * per_sm;
    grid = (unsigned)(g < n_items ? g : n_items);   // (callers return early when there are no items)
    return IDL_OK;
}
// grid of a 256-thread grid-stride elementwise kernel over n elements: one thread per element, at most 16 CTAs per SM
static unsigned elementwise_grid(long long n) {
    const long long grid = (n + 255) / 256, cap = (long long)sm_count() * 16;
    return (unsigned)(grid < cap ? grid : cap);
}

// ---------------------------------------------------------------------------------------
// K6: index maps of a count matrix (SURVEY §8f rank 4): FCGR order (kmers.pyx:53-123),
// canonical (reverse-complement) folding (utils.py:191-221), normalisation of integer counts
// ---------------------------------------------------------------------------------------
// kmers.pyx:110-123: base t of a window (t = 0 oldest) contributes bit t of cgr_i / cgr_j with
// (i, j)(A, C, G, T) = (1,0) (0,0) (0,1) (1,1); the cell is (cgr_i << k) + cgr_j
IDL_HD uint32_t cgr_index(uint32_t m, int k) {
    uint32_t ci = 0, cj = 0;
    for (int t = 0; t < k; ++t) {
        const uint32_t d = (m >> (2 * (k - 1 - t))) & 3u;   // A0 C1 G2 T3, oldest base most significant
        ci |= ((~(d ^ (d >> 1))) & 1u) << t;
        cj |= (d >> 1) << t;
    }
    return (ci << k) | cj;
}
__global__ void cgr_map_kernel(const int32_t* __restrict__ counts, int32_t* __restrict__ cgr, long long total, int k, int accumulate) {
    const long long F = 1ll << (2 * k);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i >> (2 * k);
        const long long dst = row * F + cgr_index((uint32_t)(i & (F - 1)), k);
        cgr[dst] = (accumulate ? cgr[dst] : 0) + counts[i];
    }
}
// utils.py:208-221 on an integer vector: canonical k-mers (kmer <= revcomp) in increasing order, value
// int((c[kmer] + c[revcomp]) * 0.5) — the in-place float product is truncated back into the int32 array
__global__ void revcomp_fold_kernel(const int32_t* __restrict__ counts, int32_t* __restrict__ out, long long n, int k,
                                    const int32_t* __restrict__ canon, int R) {
    const long long F = 1ll << (2 * k);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n * R; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / R;
        const uint32_t kmer = (uint32_t)canon[i - row * R], rc = revcomp_index(kmer, k);
        const int a = counts[row * F + kmer], b = counts[row * F + rc];
        out[i] = (int)((double)(a + b) * 0.5);
    }
}
// counts / np.sum(counts) (utils.py:250, 272) for an int32 [n, R] matrix: one warp per row, float64 and / or float32 output
__global__ void normalize_counts_kernel(const int32_t* __restrict__ counts, long long n, int R, double* __restrict__ out64, float* __restrict__ out32) {
    const int lane = threadIdx.x & 31;
    const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    long long sum = 0;
    for (int c = lane; c < R; c += 32) sum += counts[row * R + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const double tot = (double)sum;
    for (int c = lane; c < R; c += 32) {
        const double q = (double)counts[row * R + c] / tot;
        if (out64) out64[row * R + c] = q;
        if (out32) out32[row * R + c] = (float)q;
    }
}

__global__ void rscale_kernel(const float* __restrict__ scale, float* __restrict__ rscale, int F) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < F) rscale[i] = 1.0f / scale[i];  // IEEE division: the correctly rounded reciprocal div_rn needs
}

// workspace layout: [0,24) work counters | vars | out_off | gtab | rscale   (vars / out_off / gtab only for plans too big for the
// Plan kernel parameter)
constexpr size_t WS_VARS = 64;
constexpr int MAX_VARIANTS = 4096;
constexpr int MAX_TABS = 64;
constexpr size_t WS_OUTOFF = WS_VARS + sizeof(VarDesc) * MAX_VARIANTS;
constexpr size_t WS_GTAB = WS_OUTOFF + sizeof(int64_t) * MAX_VARIANTS;
constexpr size_t WS_RSCALE = WS_GTAB + sizeof(uint32_t) * RNG_BLOCK * MAX_TABS;
constexpr size_t WS_TOTAL = WS_RSCALE + sizeof(float) * 4096;

// the instantiation of a kernel template for an output kind (nullptr for an unknown kind)
template <typename Kernel>
static Kernel kernel_for_out(int out_kind, Kernel stats, Kernel counts_i32, Kernel freq_f32, Kernel std_f32, Kernel freq_f64, Kernel canon_f32,
                             Kernel canon_std_f32, Kernel canon_f64) {
    static_assert(IDL_OUT_COUNTS_I32 == 0 && IDL_OUT_FREQ_F32 == 1 && IDL_OUT_STD_F32 == 2 && IDL_OUT_FREQ_F64 == 3 && OUT_STATS == 4, "by_kind order");
    static_assert(IDL_OUT_CANON_F32 == OUT_CANON_BIT + IDL_OUT_FREQ_F32 && IDL_OUT_CANON_STD_F32 == OUT_CANON_BIT + IDL_OUT_STD_F32 &&
                  IDL_OUT_CANON_F64 == OUT_CANON_BIT + IDL_OUT_FREQ_F64, "canonical kinds = 8 + frequency kind");
    const Kernel by_kind[] = {counts_i32, freq_f32, std_f32, freq_f64, stats};
    const Kernel canon_by_kind[] = {nullptr, canon_f32, canon_std_f32, canon_f64};
    if (out_kind >= IDL_OUT_CANON_F32 && out_kind <= IDL_OUT_CANON_F64) return canon_by_kind[out_kind - OUT_CANON_BIT];
    return out_kind >= 0 && out_kind <= OUT_STATS ? by_kind[out_kind] : nullptr;
}
// the output kinds the public entry points accept
static bool public_out_kind(int out_kind) {
    return (out_kind >= IDL_OUT_COUNTS_I32 && out_kind <= IDL_OUT_FREQ_F64) || (out_kind >= IDL_OUT_CANON_F32 && out_kind <= IDL_OUT_CANON_F64);
}

template <int K, int NT>
static int launch_profiles(const ProfParams& p, const Plan& plan, int out_kind, cudaStream_t st, int* grid_out) {
    const auto kern = kernel_for_out(out_kind, profiles_kernel<K, NT, OUT_STATS>, profiles_kernel<K, NT, IDL_OUT_COUNTS_I32>, profiles_kernel<K, NT, IDL_OUT_FREQ_F32>,
                                     profiles_kernel<K, NT, IDL_OUT_STD_F32>, profiles_kernel<K, NT, IDL_OUT_FREQ_F64>, profiles_kernel<K, NT, IDL_OUT_CANON_F32>,
                                     profiles_kernel<K, NT, IDL_OUT_CANON_STD_F32>, profiles_kernel<K, NT, IDL_OUT_CANON_F64>);
    if (!kern) return set_error(IDL_EINVAL, "unknown out_kind%s %lld", "", out_kind);
    const size_t smem = sizeof(ProfSmem<K, NT>);
    unsigned grid = 0;
    if (const int rc = persistent_grid(kern, NT, smem, p.cta_cap, p.n_items, "profiles", grid); rc != IDL_OK) return rc;
    if (grid_out) *grid_out = (int)grid;
    kern<<<grid, NT, smem, st>>>(p, plan); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

static int dispatch_k(const ProfParams& p, const Plan& plan, int k, int out_kind, cudaStream_t st, int* grid_out = nullptr) {
    switch (k) {
        case 1: return launch_profiles<1, 64>(p, plan, out_kind, st, grid_out);
        case 2: return launch_profiles<2, 64>(p, plan, out_kind, st, grid_out);
        case 3: return launch_profiles<3, 64>(p, plan, out_kind, st, grid_out);
        case 4: return launch_profiles<4, 128>(p, plan, out_kind, st, grid_out);
        case 5: return launch_profiles<5, 256>(p, plan, out_kind, st, grid_out);
        case 6: return launch_profiles<6, 512>(p, plan, out_kind, st, grid_out);
    }
    return set_error(IDL_EUNSUPPORTED, "idl_profiles: unsupported k%s", "");
}

// ---- one profile request, as the entry points receive it (what an entry point does not take stays zero) ----
struct ProfCall {
    const uint32_t* codes; const uint32_t* nmask; const int64_t* chunk_off; const int32_t* len; int64_t n_seqs_total;
    const int32_t* sidx; int64_t n_items, seq_id0; int k; const idl_variant* variants; int n_variants; const int32_t* sel; int S;
    uint64_t seed; const int64_t* edit_off; const uint32_t* edits; int out_kind; void* out; const int64_t* out_off; int64_t out_stride;
    int pseudocount, accumulate;      // accumulate: bit 0 adds to the counts, bits 8..15 cap the generic kernel's CTAs per SM
    const float* mean; const float* scale; int32_t* status; unsigned char* ws; size_t ws_bytes; cudaStream_t st;
    double* stats_partials; double* stats_n; int* n_parts;   // OUT_STATS: the generic kernel's partials, and how many it wrote
    const void* prep; size_t prep_size;                        // prepared buffer (idl_profiles_prepared)
    void* chunk; size_t chunk_size; int64_t max_long;          // chunked-path scratch (idl_profiles_chunked)
};

// a request with the arguments every entry point takes (S = n_variants: no slot selection)
static ProfCall prof_call(const uint32_t* codes, const uint32_t* nmask, const int64_t* chunk_off, const int32_t* len, int64_t n_seqs_total, const int32_t* sidx,
                          int64_t n_items, int64_t seq_id0, int k, const idl_variant* variants, int n_variants, uint64_t seed, void* ws, size_t ws_bytes, void* stream) {
    ProfCall c{};
    c.codes = codes; c.nmask = nmask; c.chunk_off = chunk_off; c.len = len; c.n_seqs_total = n_seqs_total; c.sidx = sidx;
    c.n_items = n_items; c.seq_id0 = seq_id0; c.k = k; c.variants = variants; c.n_variants = n_variants; c.S = n_variants; c.seed = seed;
    c.ws = reinterpret_cast<unsigned char*>(ws); c.ws_bytes = ws_bytes; c.st = (cudaStream_t)stream;
    return c;
}

// the checks every request starts with; `who` names the entry point in the messages
static int check_request(const ProfCall& c, const char* who) {
    if (!c.codes || !c.nmask || !c.chunk_off || !c.len || !c.variants || (!c.out && c.out_kind != OUT_STATS) || !c.out_off || !c.ws)
        return set_error(IDL_EINVAL, "%s: null pointer", who);
    if (c.ws_bytes < WS_TOTAL) return set_error(IDL_EINVAL, "%s: workspace too small (need %lld bytes)", who, (long long)WS_TOTAL);
    return IDL_OK;
}

// ---- host-side plan of one call: variant descriptors, gap tables, output offsets ----
struct HostPlan {
    Plan plan;           // what the kernels receive by value (valid when inl)
    bool inl;            // fits the kernel parameter
    int n_tabs, n_bern, n_ent;
    bool has_explicit, randn_small;   // randn_small: every Random_N slot removes <= 127 windows (the producer/consumer kernel's limit)
    int kind0;
};

static int make_plan(const char* who, const ProfCall& c, HostPlan& hp) {
    static thread_local VarDesc h_vars[MAX_VARIANTS];
    static thread_local uint32_t h_gtab[MAX_TABS * RNG_BLOCK];
    double tab_p[MAX_TABS];
    int n_tabs = 0;
    auto table_of = [&](double pr) -> int {
        for (int t = 0; t < n_tabs; ++t)
            if (tab_p[t] == pr) return t;
        if (n_tabs == MAX_TABS) return -1;
        tab_p[n_tabs] = pr;
        geometric_table(pr, h_gtab + n_tabs * RNG_BLOCK);
        return n_tabs++;
    };
    hp.n_bern = hp.n_ent = 0;
    hp.has_explicit = false;
    hp.randn_small = true;
    for (int v = 0; v < c.n_variants; ++v) {
        const idl_variant& iv = c.variants[v];
        VarDesc& d = h_vars[v];
        d.kind = iv.kind; d.rng_id = iv.rng_id; d.n_bp = iv.n_bp; d.explicit_idx = iv.explicit_idx; d.tab1 = 0; d.tab2 = 0;
        d.slope1 = 0.f; d.slope2 = 0.f;
        if (iv.kind < IDL_KIND_CLEAN || iv.kind > IDL_KIND_EXPLICIT) return set_error(IDL_EINVAL, "%s: bad variant kind %lld", who, iv.kind);
        if (iv.kind == IDL_KIND_TRANSITION || iv.kind == IDL_KIND_BOTH) {
            if (!(iv.p1 >= 0.0 && iv.p1 <= 1.0)) return set_error(IDL_EINVAL, "%s: p1 out of range", who, 0);
            d.tab1 = table_of(iv.p1); d.slope1 = gap_slope(iv.p1);
        }
        if (iv.kind == IDL_KIND_TRANSVERSION || iv.kind == IDL_KIND_BOTH) {
            if (!(iv.p2 >= 0.0 && iv.p2 <= 1.0)) return set_error(IDL_EINVAL, "%s: p2 out of range", who, 0);
            d.tab2 = table_of(iv.p2); d.slope2 = gap_slope(iv.p2);
        }
        if (d.tab1 < 0 || d.tab2 < 0) return set_error(IDL_EUNSUPPORTED, "%s: too many distinct mutation rates", who, 0);
        if (iv.kind == IDL_KIND_RANDOM_N && (iv.n_bp < 0 || iv.n_bp > LIST_CAP / 2)) return set_error(IDL_EUNSUPPORTED, "%s: Random_N n_bp must be <= 1024", who, 0);
        if (iv.kind == IDL_KIND_EXPLICIT && (!c.edit_off || !c.edits)) return set_error(IDL_EINVAL, "%s: explicit variant without edit lists", who, 0);
        if (iv.kind == IDL_KIND_EXPLICIT) hp.has_explicit = true;
        else if (iv.kind == IDL_KIND_RANDOM_N) { if (iv.n_bp * PC_K > 127) hp.randn_small = false; else if (iv.n_bp > 0) hp.n_ent += iv.n_bp; }
        else if (iv.kind != IDL_KIND_CLEAN) ++hp.n_bern;
    }
    hp.kind0 = h_vars[0].kind;
    hp.n_tabs = n_tabs;
    hp.inl = c.n_variants <= SVARS && c.S <= SVARS && n_tabs <= STABS;
    if (hp.inl) {
        memset(&hp.plan, 0, sizeof(hp.plan));
        memcpy(hp.plan.vars, h_vars, sizeof(VarDesc) * c.n_variants);
        for (int s = 0; s < c.S; ++s) hp.plan.out_off[s] = c.out_off[s];
        memcpy(hp.plan.gtab, h_gtab, sizeof(uint32_t) * RNG_BLOCK * n_tabs);
    } else {   // big plans travel through the workspace (pageable staging: the host arrays may be reused after the calls return)
        IDL_CUDA_CHECK(cudaMemcpyAsync(c.ws + WS_VARS, h_vars, sizeof(VarDesc) * c.n_variants, cudaMemcpyHostToDevice, c.st));
        IDL_CUDA_CHECK(cudaMemcpyAsync(c.ws + WS_OUTOFF, c.out_off, sizeof(int64_t) * c.S, cudaMemcpyHostToDevice, c.st));
        if (n_tabs) IDL_CUDA_CHECK(cudaMemcpyAsync(c.ws + WS_GTAB, h_gtab, sizeof(uint32_t) * RNG_BLOCK * n_tabs, cudaMemcpyHostToDevice, c.st));
    }
    return IDL_OK;
}

// identity of a prepared buffer: FNV-1a over everything the prepared data depends on
static unsigned long long prep_stamp_of(const ProfCall& c) {
    unsigned long long h = 1469598103934665603ull;
    auto mix = [&](const void* ptr, size_t nb) {
        const unsigned char* b = reinterpret_cast<const unsigned char*>(ptr);
        for (size_t i = 0; i < nb; ++i) { h ^= b[i]; h *= 1099511628211ull; }
    };
    mix(&c.codes, sizeof(c.codes)); mix(&c.sidx, sizeof(c.sidx)); mix(&c.n_items, sizeof(c.n_items)); mix(&c.seq_id0, sizeof(c.seq_id0));
    mix(&c.seed, sizeof(c.seed)); mix(&c.pseudocount, sizeof(c.pseudocount));
    for (int v = 0; v < c.n_variants; ++v) {   // slot 0 (statistics row) and the Bernoulli slots: what the buffer holds
        const idl_variant& iv = c.variants[v];
        const bool bern = iv.kind == IDL_KIND_TRANSITION || iv.kind == IDL_KIND_TRANSVERSION || iv.kind == IDL_KIND_BOTH;
        if (v == 0 || bern) { mix(&iv.kind, sizeof(iv.kind)); mix(&iv.rng_id, sizeof(iv.rng_id)); mix(&iv.p1, sizeof(iv.p1)); mix(&iv.p2, sizeof(iv.p2)); }
    }
    return h ? h : 1ull;
}

// kernel parameters of a planned request; zeroes the work counters they point at
static int fill_params(ProfParams& p, const ProfCall& c, const HostPlan& hp) {
    IDL_CUDA_CHECK(cudaMemsetAsync(c.ws, 0, 24, c.st));   // work counter, deferred-item counter, deferred scan cursor
    memset(&p, 0, sizeof(p));
    p.codes = c.codes; p.nmask = c.nmask; p.chunk_off = c.chunk_off; p.len = c.len; p.sidx = c.sidx; p.sel = c.sel;
    p.n_items = c.n_items; p.seq_id0 = c.seq_id0; p.n_seqs_total = c.n_seqs_total; p.S = c.S; p.n_vars = c.n_variants; p.n_tabs = hp.n_tabs;
    p.vars = reinterpret_cast<const VarDesc*>(c.ws + WS_VARS);
    p.seed = c.seed; p.gtab = reinterpret_cast<const uint32_t*>(c.ws + WS_GTAB);
    p.edit_off = c.edit_off; p.edits = c.edits; p.out = c.out;
    p.out_off = reinterpret_cast<const int64_t*>(c.ws + WS_OUTOFF);
    p.out_stride = c.out_stride; p.pseudocount = c.pseudocount; p.accumulate = c.accumulate & 1; p.cta_cap = (c.accumulate >> 8) & 0xFF;
    p.mean = c.mean; p.scale = c.scale; p.status = c.status;
    p.rscale = reinterpret_cast<const float*>(c.ws + WS_RSCALE);
    p.work_counter = reinterpret_cast<unsigned long long*>(c.ws);
    p.inline_plan = hp.inl ? 1 : 0;
    p.stats_partials = c.stats_partials; p.stats_n = c.stats_n;
    return IDL_OK;
}

// ---- chunked path (chunked.cuh): scratch layout and sizing ----
struct ChunkLayout { size_t off_tiles, off_rank, off_partials, bytes, smem; int grid; };

static int chunk_dense_cap(const idl_variant* variants, int n_variants, int S) {
    int nd = 0;
    for (int v = 0; v < n_variants; ++v) {
        const int kd = variants[v].kind;
        nd += (kd == IDL_KIND_TRANSITION || kd == IDL_KIND_TRANSVERSION || kd == IDL_KIND_BOTH || kd == IDL_KIND_EXPLICIT) ? 1 : 0;
    }
    return nd < S ? nd : S;
}
static ChunkLayout chunk_layout(int64_t n_items, int64_t max_long, int nd_cap) {
    ChunkLayout l;
    memset(&l, 0, sizeof(l));
    l.smem = sizeof(ChSmem) - sizeof(int) * CH_F + sizeof(int) * CH_F * (size_t)(1 + nd_cap);
    int per_sm = 0;
    if (ensure_dyn_smem((const void*)ch_tile_kernel<6>, l.smem) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ch_tile_kernel<6>, CH_NT, l.smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return l;   // grid 0: does not fit
    }
    l.grid = sm_count() * per_sm;
    l.off_tiles = 64;
    l.off_rank = l.off_tiles + (((size_t)(n_items + 1) * 8 + 15) & ~(size_t)15);
    l.off_partials = l.off_rank + (((size_t)n_items * 4 + 15) & ~(size_t)15);
    l.bytes = l.off_partials + (size_t)(max_long + l.grid) * (size_t)(1 + nd_cap) * CH_F * sizeof(int);
    return l;
}

static int profiles_impl(const ProfCall& c) {
    if (const int rc = check_request(c, "idl_profiles"); rc != IDL_OK) return rc;
    if (c.k < 1 || c.k > 6) return set_error(IDL_EUNSUPPORTED, "idl_profiles: k must be in 1..6%s (got %lld)", "", c.k);
    if (c.n_variants < 1 || c.n_variants > MAX_VARIANTS || c.S < 1 || c.S > MAX_VARIANTS)
        return set_error(IDL_EINVAL, "idl_profiles: n_variants / S out of range%s", "");
    if (!c.sel && c.S != c.n_variants) return set_error(IDL_EINVAL, "idl_profiles: S must equal n_variants without d_sel%s", "");
    if ((c.out_kind == IDL_OUT_STD_F32 || c.out_kind == IDL_OUT_CANON_STD_F32) && (!c.mean || !c.scale))
        return set_error(IDL_EINVAL, "idl_profiles: mean/scale required%s", "");
    if ((c.accumulate & 1) && c.out_kind != IDL_OUT_COUNTS_I32) return set_error(IDL_EINVAL, "idl_profiles: accumulate only for counts%s", "");
    if (c.n_items <= 0) return IDL_OK;
    // (canonical rows are written one element at a time: any stride)
    if (c.out_stride % 4 != 0 && !is_canon(c.out_kind)) return set_error(IDL_EINVAL, "idl_profiles: out_stride must be a multiple of 4%s", "");
    if (!is_canon(c.out_kind)) {   // every kernel writes these rows as 16-byte vectors: a misaligned row would fault
        bool aligned = ((uintptr_t)c.out & 15) == 0;
        for (int s = 0; s < c.S && aligned; ++s) aligned = (c.out_off[s] & 3) == 0;
        if (!aligned) return set_error(IDL_EINVAL, "idl_profiles: d_out must be 16-byte aligned and out_off multiples of 4%s", "");
    }

    HostPlan hp;
    ProfParams p;
    if (const int rc = make_plan("idl_profiles", c, hp); rc != IDL_OK) return rc;
    if (const int rc = fill_params(p, c, hp); rc != IDL_OK) return rc;
    if (c.out_kind == IDL_OUT_STD_F32) {
        const int F = 1 << (2 * c.k);
        rscale_kernel<<<(F + 255) / 256, 256, 0, c.st>>>(c.scale, reinterpret_cast<float*>(c.ws + WS_RSCALE), F); note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
    }
    if (c.out_kind == OUT_STATS) return dispatch_k(p, hp.plan, c.k, c.out_kind, c.st, c.n_parts);
    // ---- chunked path for the long items (k = 6): tiles spread over the whole grid, exact integer reduction ----
    if (c.chunk && c.k == 6 && c.max_long > 0) {
        const int nd_cap = chunk_dense_cap(c.variants, c.n_variants, c.S);
        if (nd_cap <= CH_MAX_DENSE && !((uintptr_t)c.chunk & 15)) {
            const ChunkLayout lay = chunk_layout(c.n_items, c.max_long, nd_cap);
            if (lay.grid > 0 && c.chunk_size >= lay.bytes) {
                unsigned char* cb = reinterpret_cast<unsigned char*>(c.chunk);
                ChParams cp;
                cp.p = p;
                cp.hdr = reinterpret_cast<ChHeader*>(cb);
                cp.tile_off = reinterpret_cast<long long*>(cb + lay.off_tiles);
                cp.long_rank = reinterpret_cast<int*>(cb + lay.off_rank);
                cp.partials = reinterpret_cast<int*>(cb + lay.off_partials);
                cp.max_long = c.max_long; cp.nd_cap = nd_cap; cp.grid_tiles = lay.grid;
                ch_plan_kernel<<<1, 1024, 0, c.st>>>(cp); note_launch();
                IDL_CUDA_CHECK(cudaGetLastError());
                IDL_CUDA_CHECK(ensure_dyn_smem((const void*)ch_tile_kernel<6>, lay.smem));
                ch_tile_kernel<6><<<(unsigned)lay.grid, CH_NT, lay.smem, c.st>>>(cp, hp.plan); note_launch();
                IDL_CUDA_CHECK(cudaGetLastError());
                long long rgrid = (long long)sm_count() * 2;
                if (rgrid > c.n_items) rgrid = c.n_items;
                using ReduceKernel = void (*)(ChParams, Plan);   // (OUT_STATS requests returned above)
                const ReduceKernel reduce = kernel_for_out<ReduceKernel>(c.out_kind, nullptr, ch_reduce_kernel<6, IDL_OUT_COUNTS_I32>, ch_reduce_kernel<6, IDL_OUT_FREQ_F32>,
                                                                         ch_reduce_kernel<6, IDL_OUT_STD_F32>, ch_reduce_kernel<6, IDL_OUT_FREQ_F64>,
                                                                         ch_reduce_kernel<6, IDL_OUT_CANON_F32>, ch_reduce_kernel<6, IDL_OUT_CANON_STD_F32>,
                                                                         ch_reduce_kernel<6, IDL_OUT_CANON_F64>);
                reduce<<<(unsigned)rgrid, CH_NT, 0, c.st>>>(cp, hp.plan); note_launch();
                IDL_CUDA_CHECK(cudaGetLastError());
                p.long_overflow = &cp.hdr->overflow;   // the generic kernel skips the long items (unless the plan found more than max_long)
            }
        }
    }
    // ---- producer/consumer kernel (k = 6, float outputs, whole-schedule featurisation of PREPARED items) ----
    bool pc_ok = c.prep && c.k == 6 && (c.out_kind == IDL_OUT_FREQ_F32 || c.out_kind == IDL_OUT_STD_F32) && !c.sel && c.status && hp.inl &&
                 c.n_variants <= PC_MAXS && c.n_items >= 2LL * sm_count() && c.prep_size >= prep_bytes(c.n_items);
    if (pc_ok) {
        if (hp.has_explicit || !hp.randn_small || hp.n_bern > PC_DENSE || hp.n_ent > PC_LIST || hp.n_ent * PC_K > PC_REM) pc_ok = false;
        // TMA bulk copies: 16-byte aligned sources (the output rows are, checked above)
        if (((uintptr_t)c.codes & 15) || ((uintptr_t)c.nmask & 15) || ((uintptr_t)c.prep & 15)) pc_ok = false;
    }
    if (pc_ok) {
        p.prep = const_cast<void*>(c.prep);
        p.prep_stamp = prep_stamp_of(c);
        auto kern = c.out_kind == IDL_OUT_STD_F32 ? profiles_pc_kernel<IDL_OUT_STD_F32> : profiles_pc_kernel<IDL_OUT_FREQ_F32>;
        IDL_CUDA_CHECK(ensure_dyn_smem((const void*)kern, sizeof(PcSmem)));
        long long grid = sm_count();
        if (grid > c.n_items) grid = c.n_items;
        kern<<<(unsigned)grid, PC_NT, sizeof(PcSmem), c.st>>>(p, hp.plan); note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
        p.only_deferred = 1;   // whatever the fast kernel could not take is redone by the generic one
    }
    return dispatch_k(p, hp.plan, c.k, c.out_kind, c.st);
}

}  // namespace idl

using namespace idl;

extern "C" {

int idl_abi_version(void) { return IDL_ABI_VERSION; }
long long idl_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* idl_last_error(void) { return g_err; }

int idl_geometric_table(double p, uint32_t* out128) {
    if (!out128 || !(p >= 0.0) || !(p <= 1.0)) return set_error(IDL_EINVAL, "idl_geometric_table: bad argument%s", "");
    geometric_table(p, out128);
    return IDL_OK;
}

int idl_pack(const uint8_t* d_ascii, const int64_t* d_byte_off, int64_t n, int alphabet, int64_t max_len,
             const int64_t* d_chunk_off, uint32_t* d_codes, uint32_t* d_nmask, int32_t* d_len,
             unsigned long long* d_bad, void* stream) {
    if (n < 0 || !d_byte_off || !d_chunk_off || !d_codes || !d_nmask || !d_len || !d_bad)
        return set_error(IDL_EINVAL, "idl_pack: null pointer or negative n%s", "");
    if (max_len > 0x7fffffffLL) return set_error(IDL_EUNSUPPORTED, "idl_pack: sequences longer than 2^31-1 bases%s", "");
    long long gx = n + 1;
    const long long cap = (long long)sm_count() * 32;
    if (gx > cap) gx = cap;
    long long gy = (max_len + (32LL * PACK_NT * 8) - 1) / (32LL * PACK_NT * 8);
    if (gy < 1) gy = 1;
    if (gy > 1024) gy = 1024;
    if (gx * gy > cap * 4 && gx > 1) { gx = cap * 4 / gy; if (gx < 1) gx = 1; }
    pack_kernel<<<dim3((unsigned)gx, (unsigned)gy), PACK_NT, 0, (cudaStream_t)stream>>>(
        d_ascii, d_byte_off, d_chunk_off, n, alphabet, d_codes, d_nmask, d_len, d_bad); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

size_t idl_profiles_workspace_bytes(void) { return WS_TOTAL; }

int idl_profiles(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                 const int32_t* d_len, int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items,
                 int64_t seq_id0, int k, const idl_variant* variants, int n_variants, const int32_t* d_sel,
                 int S, uint64_t seed, const int64_t* d_edit_off, const uint32_t* d_edits, int out_kind,
                 void* d_out, const int64_t* out_off, int64_t out_stride, int pseudocount, int accumulate,
                 const float* d_mean, const float* d_scale, int32_t* d_status, void* d_workspace,
                 size_t workspace_bytes, void* stream) {
    if (!public_out_kind(out_kind)) return set_error(IDL_EINVAL, "idl_profiles: unknown out_kind%s %lld", "", out_kind);
    ProfCall c = prof_call(d_codes, d_nmask, d_chunk_off, d_len, n_seqs_total, d_sidx, n_items, seq_id0, k, variants, n_variants, seed, d_workspace, workspace_bytes, stream);
    c.sel = d_sel; c.S = S; c.edit_off = d_edit_off; c.edits = d_edits; c.out_kind = out_kind; c.out = d_out; c.out_off = out_off;
    c.out_stride = out_stride; c.pseudocount = pseudocount; c.accumulate = accumulate; c.mean = d_mean; c.scale = d_scale; c.status = d_status;
    return profiles_impl(c);
}

size_t idl_profiles_chunked_bytes(int64_t n_items, int64_t max_long_items, const idl_variant* variants, int n_variants, int S) {
    if (n_items <= 0 || max_long_items <= 0 || !variants || n_variants < 1 || S < 1) return 0;
    const int nd_cap = chunk_dense_cap(variants, n_variants, S);
    if (nd_cap > CH_MAX_DENSE) return 0;
    const ChunkLayout lay = chunk_layout(n_items, max_long_items, nd_cap);
    return lay.grid > 0 ? lay.bytes : 0;
}

int idl_profiles_chunked(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                         const int32_t* d_len, int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items,
                         int64_t seq_id0, int k, const idl_variant* variants, int n_variants, const int32_t* d_sel,
                         int S, uint64_t seed, const int64_t* d_edit_off, const uint32_t* d_edits, int out_kind,
                         void* d_out, const int64_t* out_off, int64_t out_stride, int pseudocount, int accumulate,
                         const float* d_mean, const float* d_scale, void* d_scratch, size_t scratch_bytes, int64_t max_long_items,
                         void* d_workspace, size_t workspace_bytes, void* stream) {
    if (!public_out_kind(out_kind)) return set_error(IDL_EINVAL, "idl_profiles_chunked: unknown out_kind%s %lld", "", out_kind);
    if (!d_scratch || max_long_items < 0) return set_error(IDL_EINVAL, "idl_profiles_chunked: scratch required%s", "");
    ProfCall c = prof_call(d_codes, d_nmask, d_chunk_off, d_len, n_seqs_total, d_sidx, n_items, seq_id0, k, variants, n_variants, seed, d_workspace, workspace_bytes, stream);
    c.sel = d_sel; c.S = S; c.edit_off = d_edit_off; c.edits = d_edits; c.out_kind = out_kind; c.out = d_out; c.out_off = out_off;
    c.out_stride = out_stride; c.pseudocount = pseudocount; c.accumulate = accumulate; c.mean = d_mean; c.scale = d_scale;
    c.chunk = d_scratch; c.chunk_size = scratch_bytes; c.max_long = max_long_items;
    return profiles_impl(c);
}

int idl_profiles_prepared(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                          const int32_t* d_len, int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items,
                          int64_t seq_id0, int k, const idl_variant* variants, int n_variants, uint64_t seed, int out_kind,
                          void* d_out, const int64_t* out_off, int64_t out_stride, int pseudocount,
                          const float* d_mean, const float* d_scale, int32_t* d_status, const void* d_prep, size_t prep_size,
                          void* d_workspace, size_t workspace_bytes, void* stream) {
    if (public_out_kind(out_kind) && is_canon(out_kind))
        return set_error(IDL_EINVAL, "idl_profiles_prepared: canonical output kinds are not supported (use idl_profiles or idl_profiles_chunked)%s", "");
    if (out_kind != IDL_OUT_FREQ_F32 && out_kind != IDL_OUT_STD_F32) return set_error(IDL_EINVAL, "idl_profiles_prepared: float32 outputs only%s", "");
    if (!d_prep || !d_status) return set_error(IDL_EINVAL, "idl_profiles_prepared: d_prep and d_status are required%s", "");
    ProfCall c = prof_call(d_codes, d_nmask, d_chunk_off, d_len, n_seqs_total, d_sidx, n_items, seq_id0, k, variants, n_variants, seed, d_workspace, workspace_bytes, stream);
    c.out_kind = out_kind; c.out = d_out; c.out_off = out_off; c.out_stride = out_stride; c.pseudocount = pseudocount;
    c.mean = d_mean; c.scale = d_scale; c.status = d_status; c.prep = d_prep; c.prep_size = prep_size;
    return profiles_impl(c);
}

size_t idl_prepare_bytes(int64_t n_items) { return n_items > 0 ? prep_bytes(n_items) : 0; }

int idl_profiles_prepare(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off, const int32_t* d_len,
                         int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items, int64_t seq_id0, int k,
                         const idl_variant* variants, int n_variants, uint64_t seed, int pseudocount, void* d_prep, size_t prep_size,
                         double* d_partials, double* d_part_n, int max_parts, int* n_parts, int32_t* d_status, void* d_workspace,
                         size_t workspace_bytes, void* stream) {
    int64_t offs[PC_MAXS] = {};   // the prepare pass writes no profile rows
    ProfCall c = prof_call(d_codes, d_nmask, d_chunk_off, d_len, n_seqs_total, d_sidx, n_items, seq_id0, k, variants, n_variants, seed, d_workspace, workspace_bytes, stream);
    c.out_kind = OUT_STATS; c.out_off = offs; c.pseudocount = pseudocount; c.status = d_status;
    if (!d_prep || !d_status) return set_error(IDL_EINVAL, "idl_profiles_prepare: null pointer%s", "");
    if (const int rc = check_request(c, "idl_profiles_prepare"); rc != IDL_OK) return rc;
    if (k != PC_K) return set_error(IDL_EUNSUPPORTED, "idl_profiles_prepare: k must be 6%s (got %lld)", "", k);
    if (n_variants < 1 || n_variants > PC_MAXS) return set_error(IDL_EUNSUPPORTED, "idl_profiles_prepare: 1..64 variants%s", "");
    if (n_items <= 0) { if (n_parts) *n_parts = 0; return IDL_OK; }
    if (prep_size < prep_bytes(n_items)) return set_error(IDL_EINVAL, "idl_profiles_prepare: d_prep too small%s (need %lld bytes)", "", (long long)prep_bytes(n_items));
    if (((uintptr_t)d_prep & 15) || ((uintptr_t)d_codes & 15) || ((uintptr_t)d_nmask & 7)) return set_error(IDL_EINVAL, "idl_profiles_prepare: misaligned buffer%s", "");
    if (d_partials && (!d_part_n || !n_parts || max_parts < sm_count() * 8)) return set_error(IDL_EINVAL, "idl_profiles_prepare: statistics need d_part_n, n_parts and max_parts >= 8 x SMs%s", "");
    HostPlan hp;
    if (const int rc = make_plan("idl_profiles_prepare", c, hp); rc != IDL_OK) return rc;
    if (!hp.inl || hp.has_explicit || hp.n_bern > PC_DENSE) return set_error(IDL_EUNSUPPORTED, "idl_profiles_prepare: at most 3 Bernoulli slots, 4 distinct rates, no explicit lists%s", "");
    if (hp.kind0 == IDL_KIND_RANDOM_N && variants[0].n_bp > 0) return set_error(IDL_EUNSUPPORTED, "idl_profiles_prepare: slot 0 must be clean or a Bernoulli mimic%s", "");
    ProfParams p;
    if (const int rc = fill_params(p, c, hp); rc != IDL_OK) return rc;
    p.prep = d_prep;
    p.prep_stamp = prep_stamp_of(c);
    unsigned grid = 0;
    if (const int rc = persistent_grid(prep_kernel<PC_K>, PR_NT, sizeof(PrSmem), 0, n_items, "prepare", grid); rc != IDL_OK) return rc;
    prep_kernel<PC_K><<<grid, PR_NT, sizeof(PrSmem), c.st>>>(p, hp.plan); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    if (!d_partials) {   // no statistics wanted: nobody consumes the "left to the generic kernel" marks of this call (the prepared records keep them)
        IDL_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int32_t) * (size_t)n_items, c.st));
        return IDL_OK;
    }
    // ---- statistics of slot 0: column sums over the prepared rows + the generic kernel for the items the prepare pass left out ----
    int parts = sm_count() * 2;
    if (parts > n_items) parts = (int)n_items;
    const int rows_per_part = (int)((n_items + parts - 1) / parts);
    parts = (int)((n_items + rows_per_part - 1) / rows_per_part);
    const auto colstats = pseudocount > 0 ? colstats16_kernel<true> : colstats16_kernel<false>;   // true: every frequency is a positive normal float
    colstats<<<dim3(PC_F / 4 / CS16_NT, (unsigned)parts), CS16_NT, 0, c.st>>>(reinterpret_cast<const unsigned char*>(d_prep), n_items, rows_per_part, pseudocount,
                                                                           d_partials, d_part_n); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    p.only_deferred = 1; p.S = 1; p.n_vars = 1;
    p.stats_partials = d_partials + (size_t)parts * 2 * PC_F;
    p.stats_n = d_part_n + parts;
    int g2 = 0;
    const int rc = dispatch_k(p, hp.plan, k, OUT_STATS, c.st, &g2);
    *n_parts = parts + g2;
    return rc;
}

int idl_profile_stats(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off, const int32_t* d_len,
                      int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items, int64_t seq_id0, int k,
                      const idl_variant* variant, uint64_t seed, const int64_t* d_edit_off, const uint32_t* d_edits, int pseudocount,
                      double* d_partials, double* d_part_n, int max_parts, int* n_parts, int32_t* d_status, void* d_workspace,
                      size_t workspace_bytes, void* stream) {
    if (!d_partials || !d_part_n || !n_parts || !variant) return set_error(IDL_EINVAL, "idl_profile_stats: null pointer%s", "");
    if (max_parts < sm_count() * 8) return set_error(IDL_EINVAL, "idl_profile_stats: max_parts too small%s (need %lld)", "", (long long)sm_count() * 8);
    *n_parts = 0;
    if (n_items <= 0) return IDL_OK;
    const int64_t zero_off = 0;
    ProfCall c = prof_call(d_codes, d_nmask, d_chunk_off, d_len, n_seqs_total, d_sidx, n_items, seq_id0, k, variant, 1, seed, d_workspace, workspace_bytes, stream);
    c.edit_off = d_edit_off; c.edits = d_edits; c.out_kind = OUT_STATS; c.out_off = &zero_off; c.pseudocount = pseudocount; c.status = d_status;
    c.stats_partials = d_partials; c.stats_n = d_part_n; c.n_parts = n_parts;
    return profiles_impl(c);
}

int idl_kmer_counts(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                    const int32_t* d_len, int64_t n, int k, int32_t* d_counts, int accumulate,
                    void* d_workspace, size_t workspace_bytes, void* stream) {
    if (k < 1 || k > 6) return set_error(IDL_EUNSUPPORTED, "idl_kmer_counts: k must be in 1..6%s (got %lld)", "", k);
    const idl_variant clean{IDL_KIND_CLEAN};
    const int64_t off0 = 0;
    ProfCall c = prof_call(d_codes, d_nmask, d_chunk_off, d_len, n, nullptr, n, 0, k, &clean, 1, 0, d_workspace, workspace_bytes, stream);
    c.out_kind = IDL_OUT_COUNTS_I32; c.out = d_counts; c.out_off = &off0; c.out_stride = (int64_t)1 << (2 * k); c.accumulate = accumulate;
    return profiles_impl(c);
}

int idl_colstats_parts(int64_t n) { return n > 0 ? (int)((n + cs_rows(n) - 1) / cs_rows(n)) : 0; }

int idl_colstats(const void* d_x, int is_f64, int64_t n, int F, double* d_partials, double* d_part_n, void* stream) {
    if (!d_x || !d_partials || !d_part_n || n <= 0 || F <= 0) return set_error(IDL_EINVAL, "idl_colstats: bad argument%s", "");
    const dim3 grid((F + CS_NT - 1) / CS_NT, (unsigned)idl_colstats_parts(n));
    if (is_f64) colstats_kernel<double><<<grid, CS_NT, 0, (cudaStream_t)stream>>>((const double*)d_x, n, F, cs_rows(n), d_partials, d_part_n);
    else colstats_kernel<float><<<grid, CS_NT, 0, (cudaStream_t)stream>>>((const float*)d_x, n, F, cs_rows(n), d_partials, d_part_n);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_scaler_finalize(const double* d_partials, const double* d_part_n, int n_parts, int F, double* d_mean64,
                        double* d_var64, double* d_scale64, float* d_mean32, float* d_scale32, void* stream) {
    if (!d_partials || !d_part_n || n_parts <= 0 || F <= 0) return set_error(IDL_EINVAL, "idl_scaler_finalize: bad argument%s", "");
    scaler_finalize_kernel<<<(F + SF_COLS - 1) / SF_COLS, SF_NT, 0, (cudaStream_t)stream>>>(d_partials, d_part_n, n_parts, F, d_mean64, d_var64,
                                                                              d_scale64, d_mean32, d_scale32); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_standardize_f32(const float* d_x, float* d_out, int64_t n, int F, const float* d_mean32, const float* d_scale32,
                        void* stream) {
    if (!d_x || !d_out || !d_mean32 || !d_scale32 || n < 0 || F <= 0) return set_error(IDL_EINVAL, "idl_standardize_f32: bad argument%s", "");
    if (n == 0) return IDL_OK;
    const bool aligned16 = ((reinterpret_cast<uintptr_t>(d_x) | reinterpret_cast<uintptr_t>(d_out) | reinterpret_cast<uintptr_t>(d_mean32) |
                             reinterpret_cast<uintptr_t>(d_scale32)) & 15) == 0;
    if (F % 4 == 0 && aligned16) {
        const long long n4 = n * (F / 4);
        standardize_f32_kernel<<<elementwise_grid(n4), 256, 0, (cudaStream_t)stream>>>(d_x, d_out, n4, F / 4, d_mean32, d_scale32);
    } else {
        const long long total = n * (long long)F;
        standardize_f32_elem_kernel<<<elementwise_grid(total), 256, 0, (cudaStream_t)stream>>>(d_x, d_out, total, F, d_mean32, d_scale32);
    }
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_cgr_map(const int32_t* d_counts, int64_t n, int k, int32_t* d_cgr, int accumulate, void* stream) {
    if (!d_counts || !d_cgr || n < 0 || k < 1 || k > 12) return set_error(IDL_EINVAL, "idl_cgr_map: bad argument%s", "");
    const long long total = n << (2 * k);
    if (total == 0) return IDL_OK;
    cgr_map_kernel<<<elementwise_grid(total), 256, 0, (cudaStream_t)stream>>>(d_counts, d_cgr, total, k, accumulate); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_revcomp_canonical(int k, int32_t* h_index) {
    if (k < 1 || k > 12) return -1;
    int R = 0;
    for (uint32_t m = 0; m < (1u << (2 * k)); ++m)
        if (m <= revcomp_index(m, k)) { if (h_index) h_index[R] = (int32_t)m; ++R; }
    return R;
}

int idl_revcomp_fold(const int32_t* d_counts, int64_t n, int k, const int32_t* d_canon, int R, int32_t* d_out, void* stream) {
    if (!d_counts || !d_out || !d_canon || n < 0 || k < 1 || k > 12 || R < 1) return set_error(IDL_EINVAL, "idl_revcomp_fold: bad argument%s", "");
    if (n == 0) return IDL_OK;
    revcomp_fold_kernel<<<elementwise_grid(n * R), 256, 0, (cudaStream_t)stream>>>(d_counts, d_out, n, k, d_canon, R); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_normalize_counts(const int32_t* d_counts, int64_t n, int R, double* d_out64, float* d_out32, void* stream) {
    if (!d_counts || (!d_out64 && !d_out32) || n < 0 || R < 1) return set_error(IDL_EINVAL, "idl_normalize_counts: bad argument%s", "");
    if (n == 0) return IDL_OK;
    const long long grid = (n * 32 + 255) / 256;
    normalize_counts_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_counts, n, R, d_out64, d_out32); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_standardize_f64(const double* d_x, double* d_out64, float* d_out32, int64_t n, int F, const double* d_mean64,
                        const double* d_scale64, void* stream) {
    if (!d_x || (!d_out64 && !d_out32) || !d_mean64 || !d_scale64 || n < 0 || F <= 0) return set_error(IDL_EINVAL, "idl_standardize_f64: bad argument%s", "");
    if (n == 0) return IDL_OK;
    const long long total = n * (long long)F;
    standardize_f64_kernel<<<elementwise_grid(total), 256, 0, (cudaStream_t)stream>>>(d_x, d_out64, d_out32, total, F, d_mean64, d_scale64); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

}  // extern "C"
