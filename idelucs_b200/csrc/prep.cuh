// idelucs_b200 — "prepare" pass of the whole-schedule featurisation (k = 6): everything the AugmentFasta
// schedule (idelucs/utils.py:330-351) needs from the Bernoulli mimics (transition / transversion / combined),
// computed ONCE per sequence by a high-occupancy kernel and handed to the consumers through a caller-owned
// scratch buffer:
//
//   * the +-1 histogram deltas of every Bernoulli ("dense") slot, as a packed list
//     (kmer | ordinal << 12 | (add ? 0x8000 : 0)) — the producer/consumer kernel (profiles_pc.cuh) TMA-loads the
//     list instead of generating the mutations itself (its producers were its bottleneck: 26 k of 41 k cycles
//     per sequence went into the Bernoulli slots);
//   * the uint16 histogram of slot 0 (t_norm, the 'true' side of every pair) and its window total — the
//     StandardScaler statistics of AugmentFasta (utils.py:354-359) are column sums over these rows
//     (colstats16_kernel: HBM-bound read of 8 KB per sequence, float64 shifted-data sums in registers),
//     so the slot-0 mutations are generated once for the statistics AND the profile pass.
//
// One CTA of 256 threads per sequence at a time, 4 CTAs per SM (51 KB of shared memory each): count the clean
// histogram into int32 bins (shared atomics), mutation masks of every (slot, 64-base block) by
// the register-only mask generator (core.cuh), CTA scan -> position-sorted edit lists -> +-1 deltas
// (apply_entry), slot 0's deltas applied to the histogram.  Sequences that do not fit (longer than
// 20 480 bases, list overflows at rates far above the reference's) are flagged (meta.flags, d_status bit 1)
// and taken by the generic kernel.  Included by kernels.cu.
#pragma once

namespace idl {

// int32 bins, 4 CTAs/SM: a uint16-pair histogram fits 5 CTAs/SM but measured slower (profiles/README.md)
constexpr int PR_NT = 256;
constexpr int PR_MINB = 4;
constexpr int PR_LIST = 2048;   // edits of all dense slots of one sequence

struct PrSmem {
    alignas(16) int hist[PC_F];               // clean histogram, then slot 0's (packed to uint16 on the way out)
    alignas(16) uint32_t sseq[2][PC_SSEQ_W];  // staged sequences (codes | mask): the next item's words arrive (cp.async) while this one is processed
    alignas(16) uint32_t list[PR_LIST + 8];
    alignas(16) uint16_t delta[PC_DELTA];
    uint32_t gtabs[STABS][RNG_BLOCK];
    VarDesc dvar[PC_DENSE];
    int seg_off[PC_DENSE + 1];
    int wsum[2][PR_NT / 32];                  // edits per warp of a generation round (double-buffered: one barrier per round)
    int dtot[PC_DENSE];
    int nvalid, n_delta;
    int nd, slot0_dense;
};

__device__ __forceinline__ void cp_async16(void* sdst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(void* sdst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// counts the windows ending in the 16-base code word u of a staged sequence (idelucs/kmers.pyx:36-47) with shared atomics
// (ATOMS.POPC.INC); returns how many were counted.  Thread <-> word: a 10 kb sequence is 628 work items (2.5 rounds of 256 threads).
__device__ __forceinline__ void pr_bump(int* hist, uint32_t kmer, int d) { atomicAdd(&hist[kmer], d); }
template <int K>
__device__ __forceinline__ int pr_count_word(const uint32_t* codes, const uint32_t* nmask, int u, int* hist) {
    constexpr uint32_t KMASK = (1u << (2 * K)) - 1u;
    const uint32_t w = codes[u], prev = u > 0 ? codes[u - 1] : 0u;
    const uint32_t m = nmask[u >> 1], mprev = u > 1 ? nmask[(u >> 1) - 1] : 0xFFFFFFFFu;   // sequence start = preceded by resets (kmers.pyx:14)
    const uint64_t flags = ((uint64_t)mprev << 32) | (uint64_t)m;   // bit 31-j of m = reset flag of base j of the half-chunk
    uint64_t inv64 = flags;
#pragma unroll
    for (int d = 1; d < K; ++d) inv64 |= flags >> d;                // a window is void if any of its K bases is a reset
    const uint32_t inv = (uint32_t)(inv64 >> ((u & 1) ? 0 : 16)) & 0xFFFFu;   // bit 15-j = window ending at base j of this word
    if (inv == 0u) {   // the common case: no reset near the word, 16 unconditional updates
#pragma unroll
        for (int j = 0; j < 16; ++j) pr_bump(hist, funnel_r(w, prev, 30 - 2 * j) & KMASK, 1);
        return 16;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (!((inv >> (15 - j)) & 1u)) pr_bump(hist, funnel_r(w, prev, 30 - 2 * j) & KMASK, 1);
    return __popc(~inv & 0xFFFFu);
}

struct PrItem { int L; long long c0; uint32_t seq_id; };

template <int K>
__global__ void __launch_bounds__(PR_NT, PR_MINB) prep_kernel(const ProfParams p, const __grid_constant__ Plan plan) {
    static_assert(K == PC_K, "the prepare pass is specialised for k = 6");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PrSmem& sm = *reinterpret_cast<PrSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const long long n = p.n_items, G = gridDim.x;
    unsigned char* prep = reinterpret_cast<unsigned char*>(p.prep);
    PrepMeta* meta = reinterpret_cast<PrepMeta*>(prep + prep_meta_off());
    uint4* hist_out = reinterpret_cast<uint4*>(prep + prep_hist_off(n));
    uint4* delta_out = reinterpret_cast<uint4*>(prep + prep_delta_off(n));
    const VarDesc* gvars = p.inline_plan ? plan.vars : p.vars;

    if (tid == 0) {
        int nd = 0;
        for (int s = 0; s < p.n_vars; ++s) {
            const VarDesc vd = gvars[s];
            if (vd.kind == KIND_TRANSITION || vd.kind == KIND_TRANSVERSION || vd.kind == KIND_BOTH) {
                if (nd < PC_DENSE) sm.dvar[nd] = vd;
                ++nd;
            }
        }
        sm.nd = nd <= PC_DENSE ? nd : PC_DENSE;   // (the host refuses more dense slots than PC_DENSE)
        const int k0 = gvars[0].kind;
        sm.slot0_dense = (k0 == KIND_TRANSITION || k0 == KIND_TRANSVERSION || k0 == KIND_BOTH) ? 1 : 0;
        if (blockIdx.x == 0) {
            PrepHeader h;
            h.stamp = p.prep_stamp; h.n_items = n; h.n_dense = sm.nd; h.slot0_dense = sm.slot0_dense;
            for (int i = 0; i < 10; ++i) h.pad[i] = 0;
            *reinterpret_cast<PrepHeader*>(prep) = h;
        }
    }
    for (int i = tid; i < STABS * RNG_BLOCK; i += PR_NT)
        (&sm.gtabs[0][0])[i] = i < p.n_tabs * RNG_BLOCK ? (p.inline_plan ? (&plan.gtab[0][0])[i] : p.gtab[i]) : 0u;
    auto table = [&](int t) -> const uint32_t* { return t < STABS ? sm.gtabs[t] : p.gtab + t * RNG_BLOCK; };

    // Items are assigned statically (item = blockIdx.x + j * gridDim.x), so the next item is known at once: its metadata is
    // loaded two iterations ahead and its packed words are copied global -> shared asynchronously (cp.async, no registers)
    // while the current item is processed — no global-memory latency on the per-item critical path.
    auto item_of = [&](long long j) { return (long long)blockIdx.x + j * G; };
    auto load_item = [&](long long item) {
        PrItem it;
        it.L = -1; it.c0 = 0; it.seq_id = 0u;
        if (item < n) {
            const long long seq = p.sidx ? (long long)__ldg(p.sidx + item) : item;
            it.L = __ldg(p.len + seq);
            it.c0 = __ldg(reinterpret_cast<const long long*>(p.chunk_off) + seq);
            it.seq_id = (uint32_t)(p.seq_id0 + seq);
        }
        return it;
    };
    auto chunks_of = [](int L) { return (L + CHUNK_BASES - 1) / CHUNK_BASES; };
    auto issue_copy = [&](int buf, const PrItem& it) {
        const int nch = chunks_of(it.L);
        if (it.L > 0 && nch <= SSEQ_CHUNKS) {
            const unsigned char* gc = reinterpret_cast<const unsigned char*>(p.codes + it.c0 * 4);
            const unsigned char* gm = reinterpret_cast<const unsigned char*>(p.nmask + it.c0 * 2);
            unsigned char* sc = reinterpret_cast<unsigned char*>(sm.sseq[buf]);
            unsigned char* smk = reinterpret_cast<unsigned char*>(sm.sseq[buf] + SSEQ_CW);
            for (int c = tid; c < nch; c += PR_NT) {
                cp_async16(sc + c * 16, gc + c * 16);
                cp_async8(smk + c * 8, gm + c * 8);
            }
        }
        cp_async_commit();
    };
    PrItem cur = load_item(item_of(0)), nxt = load_item(item_of(1));
    issue_copy(0, cur);
    for (long long j = 0;; ++j) {
        const long long item = item_of(j);
        if (item >= n) break;
        const int buf = (int)(j & 1);
        const PrItem nn = load_item(item_of(j + 2));   // registers; first used one iteration later
        __syncthreads();                               // everybody is done with item j-1 (shared buffers, the other sseq half)
        issue_copy(buf ^ 1, nxt);                      // item j+1: lands during this iteration
        if (tid == 0) {
            sm.nvalid = 0; sm.n_delta = 0;
            for (int q = 0; q < PC_DENSE; ++q) sm.dtot[q] = 0;
        }
        for (int i = tid; i < (int)(sizeof(sm.hist) / 16); i += PR_NT) reinterpret_cast<uint4*>(sm.hist)[i] = make_uint4(0u, 0u, 0u, 0u);
        const int L = cur.L;
        const uint32_t seq_id = cur.seq_id;
        const int nchunks = chunks_of(L);
        const int nd = sm.nd;
        const bool slot0_dense = sm.slot0_dense != 0;
        bool defer = nchunks > SSEQ_CHUNKS;
        uint32_t* codes = sm.sseq[buf];
        uint32_t* nmask = sm.sseq[buf] + SSEQ_CW;
        cp_async_wait<1>();                            // this thread's copies of item j have landed
        if (!defer) {
            if (tid < 4) codes[nchunks * 4 + tid] = 0u;           // slack chunk (window reads run one word past the end)
            if (tid < 2) nmask[nchunks * 2 + tid] = 0xFFFFFFFFu;
        }
        __syncthreads();                               // ... and everybody else's; histogram cleared
        if (!defer) {
            // ---- clean histogram (idelucs/kmers.pyx:38-50) ----
            {
                int nv = 0;
                for (int u = tid; u < nchunks * 4; u += PR_NT) nv += pr_count_word<K>(codes, nmask, u, sm.hist);
                nv = warp_sum(nv);
                if (lane == 0 && nv) atomicAdd(&sm.nvalid, nv);
            }
            // ---- mutation masks of every (dense slot, block), position-sorted edit lists (slot-major).  Work item w =
            // ---- slot * nblocks + block; a round covers 2 * PR_NT items, warp g the 64 consecutive items from w0 + 64 g
            // ---- (two per lane, masks stay in registers), so ONE barrier per round orders the warps' list segments ----
            const int nblocks = nchunks, W = nd * nblocks;
            const int wid = tid >> 5;
            int base = 0, round = 0;
            for (int w0 = 0; w0 < W; w0 += 2 * PR_NT, ++round) {   // uniform trip count
                BlockMasks m[2];
                int cnt[2], bq[2], bb[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int w = w0 + wid * 64 + h * 32 + lane;
                    m[h].a = m[h].b = m[h].ch = 0;
                    bq[h] = 0; bb[h] = -1;
                    if (w < W) {
                        int q = 0, b = w;
                        while (b >= nblocks) { b -= nblocks; ++q; }   // (at most PC_DENSE - 1 steps)
                        const VarDesc vd = sm.dvar[q];
                        m[h] = block_masks(vd.kind, p.seed, seq_id, (uint32_t)vd.rng_id, b, L, nmask, table(vd.tab1), vd.slope1, table(vd.tab2), vd.slope2);
                        bq[h] = q; bb[h] = b;
                    }
                    cnt[h] = block_masks_count(m[h]);
                }
                int inc0 = cnt[0], inc1 = cnt[1];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t0 = __shfl_up_sync(0xffffffffu, inc0, o), t1 = __shfl_up_sync(0xffffffffu, inc1, o);
                    if (lane >= o) { inc0 += t0; inc1 += t1; }
                }
                const int tot0 = __shfl_sync(0xffffffffu, inc0, 31), tot1 = __shfl_sync(0xffffffffu, inc1, 31);
                if (lane == 0) sm.wsum[round & 1][wid] = tot0 + tot1;
                __syncthreads();
                int wbase = base, total = 0;
#pragma unroll
                for (int g = 0; g < PR_NT / 32; ++g) {
                    const int v = sm.wsum[round & 1][g];
                    if (g < wid) wbase += v;
                    total += v;
                }
                if (base + total > PR_LIST) { defer = true; break; }   // uniform
                const int off[2] = {wbase + inc0 - cnt[0], wbase + tot0 + inc1 - cnt[1]};
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (bb[h] == 0) sm.seg_off[bq[h]] = off[h];
                    if (cnt[h]) block_masks_write(m[h], bb[h], codes, sm.list + off[h]);
                }
                base += total;
            }
            if (tid == 0) sm.seg_off[nd] = base;
            __syncthreads();   // lists, seg_off and the clean histogram are complete
            if (!defer) {
                // ---- edits -> +-1 deltas (thread <-> edit, one evaluation: the deltas wait in registers for their list slot);
                // ---- slot 0's deltas also go into the histogram ----
                for (int i0 = 0; i0 < base; i0 += PR_NT) {   // uniform trip count (warp collectives inside)
                    const int i = i0 + tid;
                    int jj = 0, cnt = 0, dt = 0;
                    uint32_t d[K];
#pragma unroll
                    for (int t = 0; t < K; ++t) d[t] = 0u;
                    if (i < base) {
                        while (i >= sm.seg_off[jj + 1]) ++jj;
                        const int so = sm.seg_off[jj];
                        cnt = entry_deltas<K>(codes, nmask, L, sm.list + so, sm.seg_off[jj + 1] - so, i - so, d, &dt);
                    }
                    int inc = cnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int t = __shfl_up_sync(0xffffffffu, inc, o);
                        if (lane >= o) inc += t;
                    }
                    const int wtot = __shfl_sync(0xffffffffu, inc, 31);
                    int wbase = 0;
                    if (lane == 31 && wtot) wbase = atomicAdd(&sm.n_delta, wtot);
                    wbase = __shfl_sync(0xffffffffu, wbase, 31);
                    if (cnt && wbase + wtot <= PC_DELTA) {
                        int slot = wbase + inc - cnt;
                        const uint32_t tag = (uint32_t)jj << 12;
                        const bool to_hist = slot0_dense && jj == 0;
#pragma unroll
                        for (int t = 0; t < K; ++t) {
                            if (d[t] & 0x1000u) {
                                const uint32_t km = d[t] & 0xFFFu;
                                sm.delta[slot++] = (uint16_t)(km | tag);
                                if (to_hist) pr_bump(sm.hist, km, -1);
                            }
                            if (d[t] & 0x10000000u) {
                                const uint32_t km = (d[t] >> 16) & 0xFFFu;
                                sm.delta[slot++] = (uint16_t)(km | tag | 0x8000u);
                                if (to_hist) pr_bump(sm.hist, km, +1);
                            }
                        }
                        if (dt) atomicAdd(&sm.dtot[jj], dt);
                    }
                }
                __syncthreads();
                if (sm.n_delta > PC_DELTA) defer = true;   // uniform
            }
        }
        if (defer) {
            if (tid == 0) {
                PrepMeta mt;
                mt.n_delta = 0; mt.total0 = 0; mt.base_total = 0; mt.flags = 1; mt.pad = 0;
                for (int q = 0; q < PC_DENSE; ++q) mt.dtot[q] = 0;
                meta[item] = mt;
                if (p.status) atomicOr(p.status + item, 2);
                atomicAdd(p.work_counter + 1, 1ull);
            }
        } else {
            // ---- hand over: slot 0's histogram, the delta list, the totals ----
            const int n_delta = sm.n_delta;
            for (int i = tid; i < PC_F / 8; i += PR_NT) {   // 8 bins -> one 16-byte store of uint16 counts (every count <= 20 480)
                const int4 lo = reinterpret_cast<const int4*>(sm.hist)[2 * i], hi = reinterpret_cast<const int4*>(sm.hist)[2 * i + 1];
                hist_out[(size_t)item * (PC_F / 8) + i] = make_uint4((uint32_t)lo.x | ((uint32_t)lo.y << 16), (uint32_t)lo.z | ((uint32_t)lo.w << 16),
                                                                     (uint32_t)hi.x | ((uint32_t)hi.y << 16), (uint32_t)hi.z | ((uint32_t)hi.w << 16));
            }
            const int nq = (n_delta * 2 + 15) >> 4;
            for (int i = tid; i < nq; i += PR_NT) delta_out[(size_t)item * (PC_DELTA / 8) + i] = reinterpret_cast<const uint4*>(sm.delta)[i];
            if (tid == 0) {
                PrepMeta mt;
                mt.n_delta = n_delta;
                mt.base_total = PC_F * p.pseudocount + sm.nvalid;
                mt.total0 = mt.base_total + (slot0_dense ? sm.dtot[0] : 0);
                mt.flags = 0; mt.pad = 0;
                for (int q = 0; q < PC_DENSE; ++q) mt.dtot[q] = sm.dtot[q];
                meta[item] = mt;
            }
        }
        cur = nxt; nxt = nn;
    }
    cp_async_wait<0>();
}

// StandardScaler statistics (idelucs/utils.py:354-359) of the prepared slot-0 rows: float32(count / total) per bin
// (the same correctly rounded division as the profile kernels), float64 shifted-data sums in registers.  Thread <-> 4
// bins, CTA <-> 1024 bins x one block of rows; the rows of a part are visited in ascending order and the parts merged in
// index order (idl_scaler_finalize), so the result is run-to-run identical.  HBM-bound: 8 KB read per sequence.
// The per-row facts (float total, RN(1 / total), prepared or not) are staged in shared memory 256 rows at a time — one IEEE
// division per row and CTA instead of one per row and thread — and the int -> float / float -> double conversions are done with
// integer and FP32 instructions (exact for these operands): conversion instructions issue at a quarter of the FP64 rate and
// were what bound the first version (0.36 ms per 100 000 rows against 0.12 ms for the read).
constexpr int CS16_NT = 256;
constexpr int CS16_RC = 256;   // rows per staged chunk

template <bool NZ>
__device__ __forceinline__ double widen_pos(float q) {   // (double)q for a positive normal float q (NZ) or q = +0 (!NZ), exactly
    const uint32_t b = __float_as_uint(q);
    const uint32_t hi = (NZ || b) ? (b >> 3) + 0x38000000u : 0u;
    return __hiloint2double((int)hi, (int)(b << 29));
}
// float(c16 + pc) for a 16-bit count c16 in the low / high half of w: the byte permute builds the float 2^23 + c16 directly
// (0x4B00'xxxx), and 2^23 + c16 - (2^23 - pc) is exact
__device__ __forceinline__ float half_to_float(uint32_t w, int hi_half, float unbias) {
    return __uint_as_float(__byte_perm(w, 0x4B000000u, hi_half ? 0x7432 : 0x7410)) - unbias;
}

template <bool NZ>
__global__ void __launch_bounds__(CS16_NT) colstats16_kernel(const unsigned char* __restrict__ prep, long long n, int rows_per_part, int pseudocount,
                                                              double* __restrict__ partials, double* __restrict__ part_n) {
    __shared__ float s_tot[CS16_RC], s_y[CS16_RC];   // s_tot < 0: the row was not prepared (the generic kernel's parts cover it)
    __shared__ int s_first;
    const int vec = blockIdx.x * CS16_NT + threadIdx.x;   // 4-bin granule
    const long long r0 = (long long)blockIdx.y * rows_per_part;
    const long long r1 = r0 + rows_per_part < n ? r0 + rows_per_part : n;
    const int4* meta = reinterpret_cast<const int4*>(prep + prep_meta_off());   // first half of PrepMeta: n_delta, total0, base_total, flags
    const uint2* hist = reinterpret_cast<const uint2*>(prep + prep_hist_off(n)) + vec;
    const float unbias = 8388608.0f - (float)pseudocount;
    auto row_q = [&](uint2 pk, float ftot, float y, double (&q)[4]) {
        q[0] = widen_pos<NZ>(div_rn(half_to_float(pk.x, 0, unbias), ftot, y));
        q[1] = widen_pos<NZ>(div_rn(half_to_float(pk.x, 1, unbias), ftot, y));
        q[2] = widen_pos<NZ>(div_rn(half_to_float(pk.y, 0, unbias), ftot, y));
        q[3] = widen_pos<NZ>(div_rn(half_to_float(pk.y, 1, unbias), ftot, y));
    };
    // the shift of the shifted-data sums = the part's first prepared row
    if (threadIdx.x == 0) s_first = 0x7fffffff;
    __syncthreads();
    for (long long r = r0 + threadIdx.x; r < r1; r += CS16_NT)
        if (__ldg(meta + r * 2).w == 0) { atomicMin(&s_first, (int)(r - r0)); break; }
    __syncthreads();
    double a1[4] = {0.0, 0.0, 0.0, 0.0}, a2[4] = {0.0, 0.0, 0.0, 0.0}, shift[4] = {0.0, 0.0, 0.0, 0.0};
    if (s_first != 0x7fffffff) {
        const long long rf = r0 + s_first;
        const float ftot = (float)__ldg(meta + rf * 2).y;
        row_q(__ldg(hist + rf * (PC_F / 4)), ftot, 1.0f / ftot, shift);
    }
    int cnt = 0;
    constexpr int U = 8;   // rows in flight per thread
    for (long long c0 = r0; c0 < r1; c0 += CS16_RC) {
        const int m = (int)(r1 - c0 < CS16_RC ? r1 - c0 : CS16_RC);
        __syncthreads();
        if ((int)threadIdx.x < m) {
            const int4 mt = __ldg(meta + (c0 + threadIdx.x) * 2);
            const float ftot = mt.w != 0 ? -1.f : (float)mt.y;
            s_tot[threadIdx.x] = ftot;
            s_y[threadIdx.x] = 1.0f / ftot;
        }
        __syncthreads();
        for (int i0 = 0; i0 < m; i0 += U) {
            uint2 pk[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = i0 + u < m ? i0 + u : m - 1;
                pk[u] = __ldg(hist + (c0 + i) * (PC_F / 4));
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (i0 + u >= m) continue;               // uniform over the CTA
                const float ftot = s_tot[i0 + u];
                if (ftot < 0.f) continue;                // uniform over the CTA
                double q[4];
                row_q(pk[u], ftot, s_y[i0 + u], q);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const double dd = q[e] - shift[e];
                    a1[e] += dd;
                    a2[e] = fma(dd, dd, a2[e]);
                }
                ++cnt;
            }
        }
    }
    if (vec == 0) part_n[blockIdx.y] = (double)cnt;
    const double m = cnt > 0 ? (double)cnt : 1.0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        partials[((size_t)blockIdx.y * 2 + 0) * PC_F + vec * 4 + e] = shift[e] + a1[e] / m;
        partials[((size_t)blockIdx.y * 2 + 1) * PC_F + vec * 4 + e] = a2[e] - a1[e] * a1[e] / m;
    }
}

}  // namespace idl
