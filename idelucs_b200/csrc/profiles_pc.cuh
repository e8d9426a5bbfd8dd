// idelucs_b200 — producer/consumer variant of the profiles kernel (k = 6, float outputs).
//
// One persistent CTA of 1024 threads per SM, four roles that only meet through mbarriers:
//
//  * PRODUCERS (warps 16..31) prepare sequence i+1 into one of two shared-memory contexts: count
//    the clean histogram into packed uint16 counters, precompute the Random_N removal lists of
//    every slot, the per-slot window totals, output rows and the JOB ORDER (dense slots first,
//    then the sparse slots sorted by window total).  The +-1 delta list of the Bernoulli slots is
//    NOT generated here: the prepare pass (prep.cuh) left it in global memory and one TMA bulk
//    load per sequence brings it in for the builders.
//  * BUILDERS (warps 0..7) write finished 16 KB float rows into a ring of PC_NBUF shared-memory
//    row buffers (job j uses buffer j mod PC_NBUF).  A Random_N mimic differs from the clean
//    histogram in <= 120 of 4096 bins and every untouched bin of every variant with the same
//    window total T has the SAME output value, so a buffer is only rebuilt when the job's T
//    differs from the T of the job that used it last (the jobs are sorted by T); a Bernoulli
//    slot changes most granules and always gets its own dense row (clean + delta scratch).
//  * FIX warps (one per row buffer) make the buffer's row the job's row: they undo the <= 120
//    changed bins of the previous job and write those of the new one (4-byte shared-memory
//    stores).  The changed bins are found through a zero-based delta scratch (packed biased
//    uint8): removals are subtracted with shared atomics, then a lane claims a scratch word
//    with atomicExch (which also resets it), so duplicate k-mers in the removal list are harmless.
//  * The STORE thread writes each job's row with ONE TMA bulk copy
//    (cp.async.bulk.global.shared::cta, 16 KB): the 83 GB of output never pass through the
//    LSU instruction queue (the shared-memory traffic of the other roles is not stuck behind
//    back-pressured global stores), every global write is a full line, and nothing is ever
//    re-read or partially overwritten in L2.  It also dispatches the items (atomic counter).
//
// Items this kernel cannot take (the ones the prepare pass flagged: longer than 20 480 bases,
// list overflows) are flagged in d_status (bit 1) and redone by the generic kernel.
// Included by kernels.cu (uses its helpers).
#pragma once

namespace idl {

constexpr int PC_NT = 1024, PC_HALF = 512;
constexpr int PC_K = 6, PC_F = 4096, PC_VEC = 1024, PC_PRIVW = 2048;
constexpr int PC_NBLD = 256;       // builder threads (warps 0..7)
constexpr int PC_NFIX = 224;       // fix threads (warps 8..14); warp 15 lane 0 is the store thread
constexpr int PC_NBUF = 4;         // 16 KB row buffers
constexpr int PC_NOTH = 1;         // row buffers that take the "other" jobs (dense rows, minority window totals) while the rest stream the main total
constexpr int PC_INFL = PC_NBUF - 2;   // bulk copies kept in flight besides the one just issued
constexpr int PC_FIXW = PC_NFIX / 32;   // fix warps: each owns a 4 KB scratch (biased uint8 deltas) and handles whole jobs
constexpr int PC_SCRW = 1024;      // words of one fix-warp scratch (four bins per word)
constexpr uint32_t PC_BIAS4 = 0x80808080u;
constexpr int PC_SSEQ_W = SSEQ_CW + SSEQ_MW + 6;   // staged sequence: codes | mask (+ 16-byte alignment shift and round-up)
constexpr int PC_QRING = 8;        // dispatched items buffered ahead of the producers
constexpr uint32_t PC_BIAS2 = 0x80008000u;
constexpr int PC_MAXS = 64;        // variant slots per sequence
constexpr int PC_REM = 5888;       // removed k-mers of all Random_N slots of one sequence (51 x 20 x 6 = 6120)
constexpr int PC_DELTA = 5120;     // Bernoulli +-1 deltas of one sequence
constexpr int PC_LIST = 1024;      // Random_N draws of all slots of one sequence (PC_REM / K bounds them anyway)
constexpr int PC_MAXB = 8;         // Bernoulli slots per sequence (producer tables)
constexpr int PC_DENSE = 3;        // ... of which the builders can take (one delta scratch each; the reference schedule has 3)

// ---- layout of the prepared buffer (written by prep_kernel, prep.cuh) ----
struct alignas(16) PrepMeta {              // 32 bytes per item
    int n_delta;                           // entries of the item's delta list
    int total0;                            // window total of slot 0, pseudocount included (the statistics row)
    int base_total;                        // clean window total, pseudocount included
    int flags;                             // != 0: not prepared (generic kernel takes the item)
    int dtot[PC_DENSE];                    // change of the window total per dense ordinal
    int pad;
};
static_assert(sizeof(PrepMeta) == 32, "PrepMeta layout");

struct PrepHeader {                        // 64 bytes
    unsigned long long stamp;              // identifies (items, variants, seed, ...) the buffer was prepared for
    long long n_items;
    int n_dense, slot0_dense;
    int pad[10];
};
static_assert(sizeof(PrepHeader) == 64, "PrepHeader layout");

constexpr size_t PREP_HIST_BYTES = (size_t)PC_F * 2;          // uint16 histogram of slot 0
constexpr size_t PREP_DELTA_BYTES = (size_t)PC_DELTA * 2;     // delta list (fixed stride)
__host__ __device__ inline size_t prep_meta_off() { return sizeof(PrepHeader); }
__host__ __device__ inline size_t prep_hist_off(long long n) { return sizeof(PrepHeader) + sizeof(PrepMeta) * (size_t)n; }
__host__ __device__ inline size_t prep_delta_off(long long n) { return prep_hist_off(n) + PREP_HIST_BYTES * (size_t)n; }
__host__ __device__ inline size_t prep_bytes(long long n) { return prep_delta_off(n) + PREP_DELTA_BYTES * (size_t)n + 16; }

struct alignas(16) PcCtx {
    uint2 clean16[PC_VEC];         // packed clean histogram
    uint16_t rem[PC_REM];          // Random_N: removed k-mers, slot s at [rem_off[s]*K, +nbp*K), 0xFFFF = unused
    int dtot[PC_MAXS];             // change of the counted-window total per slot
    float2 gy[PC_MAXS];            // per slot: (float total, RN(1/total))
    long long grow[PC_MAXS];       // per slot: byte offset of the output row
    unsigned long long job_dst[PC_MAXS];   // job j: byte offset of its output row | 1 when the job needs a new row
    unsigned char job_slot[PC_MAXS];   // job j -> slot: dense slots first (slot order), then sparse/clean slots by total
    unsigned char job_build[PC_MAXS];  // job j needs a rebuilt row (dense, or its total differs from job j - PC_NBUF's)
    int n_dense;
    int n_delta;
    int delta_phase;               // parity of the delta buffer's TMA load (valid when n_delta > 0)
    int defer;                     // item must be redone by the generic kernel
    int base_total;
    long long item;                // -1: no more work
};

struct PcSmem {
    PcCtx ctx[2];
    ProfParams params;             // the producers (an out-of-line function) read the launch parameters from here, not from a local-memory copy
    alignas(16) float rowbuf[PC_NBUF][PC_F];
    // scaler statistics (launch constants; global loads take ~3k cycles under the saturated write stream)
    alignas(16) float smean[PC_F];
    alignas(16) float sscale[PC_F];
    signed char srcorr[PC_F];      // RN(1/scale) = bits(MUFU.RCP(scale)) + srcorr (ulps): the exact reciprocal in 1 byte instead of 4
    int rcorr_bad;                 // a correction did not fit (never seen): every item is deferred to the generic kernel
    // producer scratch
    alignas(16) uint32_t sseq[2][PC_SSEQ_W];   // double-buffered: the TMA load of item i+1 lands while item i is prepared
    alignas(16) uint32_t list[PC_LIST + 8];
    alignas(16) uint16_t delta[2][PC_DELTA];   // Bernoulli deltas of the sequences of the two contexts (TMA-loaded from the prepared buffer): kmer | ordinal << 12 | (add ? 0x8000 : 0)
    unsigned char m_sorted[PC_MAXS];   // slots sorted by job key (dense first, then window total)
    unsigned char m_lt[PC_MAXS], m_eq[PC_MAXS];   // per slot: slots with a smaller key / with the same key
    unsigned m_exh[2];             // ballots of "the list this position wants is exhausted"
    int nvalid;
    int prep_bad;                  // the prepared buffer does not belong to this call (stamp mismatch): every item is deferred
    long long q_item[PC_QRING], q_seq[PC_QRING], q_c0[PC_QRING];   // dispatch ring written by the store thread: item, sequence, first chunk, length
    int q_len[PC_QRING];
    int4 q_meta0[PC_QRING], q_meta1[PC_QRING];   // ... and the item's PrepMeta (n_delta, total0, base_total, flags | dtot[3], pad)
    int q_head;                    // entries published so far
    // launch-uniform slot tables (built once)
    VarDesc svars[PC_MAXS];
    long long sout_off[PC_MAXS];
    int kind_class[PC_MAXS];       // 0 none, 1 Random_N, 2 Bernoulli
    int rem_off[PC_MAXS];          // first draw of the slot (x K = first rem entry)
    int nbp[PC_MAXS];
    int bern_ord[PC_MAXS];         // ordinal of a Bernoulli slot
    int bern_slot[PC_MAXB];        // slot of ordinal
    int n_bern, n_ent;
    // consumer side
    alignas(16) uint32_t dscratch[PC_DENSE][PC_PRIVW];  // dense slots (builders): biased uint16 deltas, two bins per word, one array per Bernoulli ordinal
    alignas(16) uint32_t sscratch[PC_NBUF * PC_SCRW];   // sparse jobs: one scratch per active fix warp (= per row buffer)
    // mbarriers.  Per row buffer: free (its last bulk copy has been read) -> built (builders, only when rebuilt)
    // -> full (fix warp: the row is the job's row) -> bulk copy -> free
    alignas(8) unsigned long long ctx_full[2], ctx_empty[2], row_free[PC_NBUF], row_built[PC_NBUF], row_full[PC_NBUF], seq_full[2], delta_full[2];
    int free_count[PC_NBUF];       // uses of each buffer whose bulk copy has been read.  The builders look ahead and skip the uses that
                                   // need no rebuild; an mbarrier parity wait alone can only tell adjacent phases apart
};

constexpr uint32_t PC_SUSPEND_NS = 2000u;   // upper bound of one hardware-suspended mbarrier wait (a completed phase wakes the thread at once):
                                            // long enough that waiting warps do not eat issue slots with retries
// ---- mbarrier / TMA bulk-copy primitives (sm_90+ PTX; SASS: SYNCS.*, UBLKCP) ----
__device__ __forceinline__ uint32_t smem_u32(const void* ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" ::"r"(smem_u32(bar)), "r"(parity), "r"(PC_SUSPEND_NS) : "memory");
}
// one (hardware-suspended, time-limited) wait attempt: a sleeping primitive for loops that re-check a counter
__device__ __forceinline__ void mbar_try_once(unsigned long long* bar, uint32_t parity) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n}" ::"r"(smem_u32(bar)), "r"(parity), "r"(PC_SUSPEND_NS) : "memory");
}
__device__ __forceinline__ bool mbar_test(unsigned long long* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ int ld_acquire_smem(const int* ptr) {
    int v;
    asm volatile("ld.acquire.cta.shared::cta.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(ptr)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_smem(int* ptr, int v) {
    asm volatile("st.release.cta.shared::cta.s32 [%0], %1;" ::"r"(smem_u32(ptr)), "r"(v) : "memory");
}

__device__ __forceinline__ void bar_named(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

template <int OUT>
__device__ __noinline__ void pc_producer(PcSmem& sm) {
    const ProfParams& p = sm.params;
    constexpr int K = PC_K;
    const int ptid = threadIdx.x - PC_HALF, lane = ptid & 31;
    // Items are dispatched by the store thread into a small ring (index, first chunk, length) and the
    // packed words of item A_{i+1} are TMA-loaded into the other half of sseq while A_i is prepared:
    // no global-load latency (~3k cycles under the saturated write stream) and no long-lived
    // scoreboard sits on the producers' critical path.
    auto half_count = [](int L) { return ((L + CHUNK_BASES - 1) / CHUNK_BASES) * 2; };
    auto loads_seq = [&](long long item, int L) { const int nh = half_count(L); return item < p.n_items && nh <= 2 * SSEQ_CHUNKS && nh > 0; };
    auto issue_seq_load = [&](int buf, long long item, long long c0, int L) {   // thread 0
        const int nh = half_count(L);
        if (!loads_seq(item, L)) return;
        const uint32_t shift = (uint32_t)(c0 & 1);                              // mask words start 8 bytes into a 16-byte unit
        const uint32_t cbytes = (uint32_t)nh * 8u, mbytes = ((uint32_t)nh * 4u + shift * 8u + 15u) & ~15u;
        fence_proxy_async_smem();                                               // earlier generic reads of this buffer are done
        mbar_expect_tx(&sm.seq_full[buf], cbytes + mbytes);
        bulk_load(sm.sseq[buf], p.codes + c0 * 4, cbytes, &sm.seq_full[buf]);
        bulk_load(sm.sseq[buf] + SSEQ_CW, p.nmask + c0 * 2 - shift * 2, mbytes, &sm.seq_full[buf]);
    };
    long long cur_item, cur_seq, cur_c0;
    int cur_L;
    int4 cur_m0, cur_m1;            // PrepMeta of the current item
    int n_loads0 = 0, n_loads1 = 0; // TMA loads issued into each half of sseq (mbarrier phase bookkeeping)
    int n_dloads0 = 0, n_dloads1 = 0;   // ... and into each delta buffer
    int gj0 = 0;                    // jobs of the previous (not deferred) sequences: the consumers' buffer rotation
    const unsigned char* prep_delta = reinterpret_cast<const unsigned char*>(p.prep) + prep_delta_off(p.n_items);
    while (ld_acquire_smem(&sm.q_head) < 1) __nanosleep(32);
    cur_item = sm.q_item[0]; cur_seq = sm.q_seq[0]; cur_c0 = sm.q_c0[0]; cur_L = sm.q_len[0]; cur_m0 = sm.q_meta0[0]; cur_m1 = sm.q_meta1[0];
    if (ptid == 0) issue_seq_load(0, cur_item, cur_c0, cur_L);
    int cur_phase = 0;
    if (loads_seq(cur_item, cur_L)) ++n_loads0;
    for (int it = 0;; ++it) {
        const int b = it & 1;
        PcCtx& cx = sm.ctx[b];
        while (ld_acquire_smem(&sm.q_head) < it + 2) __nanosleep(32);
        const int qs = (it + 1) & (PC_QRING - 1);
        const long long nx_item = sm.q_item[qs], nx_seq = sm.q_seq[qs], nx_c0 = sm.q_c0[qs];
        const int nx_L = sm.q_len[qs];
        const int4 nx_m0 = sm.q_meta0[qs], nx_m1 = sm.q_meta1[qs];
        if (ptid == 0) issue_seq_load(b ^ 1, nx_item, nx_c0, nx_L);            // A_{i+1}: lands during this iteration
        const int nx_phase = b ? n_loads0 : n_loads1;
        if (loads_seq(nx_item, nx_L)) { if (b) ++n_loads0; else ++n_loads1; }
        mbar_wait(&sm.ctx_empty[b], ((it >> 1) & 1) ^ 1);   // every consumer role is done with the previous occupant
        const long long item = cur_item;
        if (item >= p.n_items) {
            if (ptid == 0) { cx.item = -1; mbar_arrive(&sm.ctx_full[b]); }
            return;
        }
        const long long seq = cur_seq;
        const int L = cur_L;
        const uint32_t seq_id = (uint32_t)(p.seq_id0 + seq);
        const int nhalf = half_count(L);
        const int n_delta = sm.n_bern > 0 ? cur_m0.x : 0;
        const bool fits = nhalf <= 2 * SSEQ_CHUNKS && !sm.rcorr_bad && !sm.prep_bad && cur_m0.w == 0 && n_delta <= PC_DELTA;
        // the delta list of this sequence: one TMA bulk load into the context's delta buffer.  Every consumer role is done with
        // the buffer's previous occupant (ctx_empty above), and the copy lands while the producers prepare the rest.
        const int dphase = b ? n_dloads1 : n_dloads0;
        if (fits && n_delta > 0) {
            if (ptid == 0) {
                const uint32_t bytes = ((uint32_t)n_delta * 2u + 15u) & ~15u;
                fence_proxy_async_smem();
                mbar_expect_tx(&sm.delta_full[b], bytes);
                bulk_load(sm.delta[b], prep_delta + (size_t)item * PREP_DELTA_BYTES, bytes, &sm.delta_full[b]);
            }
            if (b) ++n_dloads1; else ++n_dloads0;
        }
        if (ptid == 0) { cx.item = item; cx.defer = fits ? 0 : 1; cx.n_delta = n_delta; cx.delta_phase = dphase & 1; sm.nvalid = 0; }
        for (int i = ptid; i < PC_MAXS; i += PC_HALF) cx.dtot[i] = 0;
        uint32_t* cw = reinterpret_cast<uint32_t*>(cx.clean16);   // two uint16 counters per word (counts <= 20 480)
        if (fits) {
            // ---- the staged sequence (TMA) -> count from shared memory ----
            uint32_t* codes_w = sm.sseq[b];
            uint32_t* nmask_w = sm.sseq[b] + SSEQ_CW + (int)(cur_c0 & 1) * 2;
            reinterpret_cast<uint4*>(cw)[ptid] = make_uint4(0u, 0u, 0u, 0u);
            if (nhalf > 0) mbar_wait(&sm.seq_full[b], cur_phase & 1);
            if (ptid < 4) codes_w[nhalf * 2 + ptid] = 0u;
            if (ptid < 2) nmask_w[nhalf + ptid] = 0xFFFFFFFFu;
            bar_named(1, PC_HALF);
            const uint32_t* codes = codes_w;
            const uint32_t* nmask = nmask_w;
            int nv = 0;
            for (int h = ptid; h < nhalf; h += PC_HALF) {
                const uint2 w = reinterpret_cast<const uint2*>(codes)[h];
                nv += count_half<K>(codes, nmask, h, w.x, w.y, [&](uint32_t kmer) { atomicAdd(&cw[kmer >> 1], 1u << ((kmer & 1u) * 16u)); });
            }
            nv = warp_sum(nv);
            if (lane == 0 && nv) atomicAdd(&sm.nvalid, nv);
            bar_named(1, PC_HALF);
            if (ptid == 0) cx.base_total = PC_F * p.pseudocount + sm.nvalid;
            // ---- Random_N slots: draws (thread <-> slot, philox call) ----
            const int n_ent = sm.n_ent;   // <= PC_LIST (host-checked)
            {
                constexpr int e0 = 0;
                for (int q = ptid; q < p.S * 8; q += PC_HALF) {
                    const int c = q >> 3, j = q & 7;
                    const int nb = sm.kind_class[c] == 1 ? sm.nbp[c] : 0;
                    const int off = sm.rem_off[c] - e0;
                    if (4 * j < nb && off >= 0 && off + nb <= PC_LIST) {
                        const U4 r = random_n_words(p.seed, seq_id, (uint32_t)sm.svars[c].rng_id, (uint32_t)j);
                        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                        for (int t = 0; t < 4; ++t)
                            if (4 * j + t < nb) sm.list[off + 4 * j + t] = random_n_entry(w[t], L) | ((uint32_t)c << 25);
                    }
                }
                bar_named(1, PC_HALF);
                constexpr uint32_t KMASK = (1u << (2 * K)) - 1u, NMASKK = (1u << K) - 1u;
                const int n_here = n_ent - e0 < PC_LIST ? n_ent - e0 : PC_LIST;
                for (int q = ptid; q < n_here; q += PC_HALF) {
                    const uint32_t me = sm.list[q];
                    const int c = (int)(me >> 25);
                    const int nb = sm.nbp[c], off = sm.rem_off[c] - e0, i = q - off;
                    const uint32_t pme = me >> 3;
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
                    uint16_t* dst = cx.rem + (sm.rem_off[c] + i) * K;
                    int cnt = 0;
                    if (!dup) {
                        const int pos = (int)(pme & 0x3FFFFFu);
                        int e_hi = pos + K - 1;
                        if (pnx != 0xFFFFFFFFu && (int)(pnx & 0x3FFFFFu) - 1 < e_hi) e_hi = (int)(pnx & 0x3FFFFFu) - 1;
                        if (L - 1 < e_hi) e_hi = L - 1;
                        const Window<K> cw = load_window<K>(codes, nmask, pos - (K - 1));
                        for (int ee = pos; ee <= e_hi; ++ee) {
                            const int sh = K - 1 - (ee - pos);
                            if (((cw.nbits >> sh) & NMASKK) == 0u) dst[cnt++] = (uint16_t)((cw.bases >> (2 * sh)) & KMASK);
                        }
                    }
                    for (int r = cnt; r < K; ++r) dst[r] = 0xFFFFu;
                    if (cnt) atomicSub(&cx.dtot[c], cnt);
                }
                bar_named(1, PC_HALF);
            }
            // ---- Bernoulli slots: their window totals come from the prepare pass ----
            if (ptid < sm.n_bern) cx.dtot[sm.bern_slot[ptid]] = ptid == 0 ? cur_m1.x : (ptid == 1 ? cur_m1.y : cur_m1.z);
            bar_named(1, PC_HALF);
        }
        if (ptid == 0 && cx.defer) { atomicOr(p.status + item, 2); atomicAdd(p.work_counter + 1, 1ull); }
        // ---- per-slot totals, output rows and the job order (dense slots first, then by window total) ----
        const int S = p.S;
        auto job_key = [&](int s) -> unsigned { return sm.kind_class[s] == 2 ? 0u : 0x40000000u | (unsigned)(cx.base_total + cx.dtot[s]); };
        {   // slots sorted by key (8 lanes per slot): rank = smaller keys + equal keys with a smaller slot index
            const int s = ptid >> 3, part = ptid & 7;
            const bool on = s < S;
            const unsigned ks = on ? job_key(s) : 0u;
            int lt = 0, eqb = 0, eq = 0;
            if (on)
                for (int t = part; t < S; t += 8) {
                    const unsigned kt = job_key(t);
                    lt += kt < ks ? 1 : 0;
                    eq += kt == ks ? 1 : 0;
                    eqb += (kt == ks && t < s) ? 1 : 0;
                }
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                lt += __shfl_xor_sync(0xffffffffu, lt, o);
                eq += __shfl_xor_sync(0xffffffffu, eq, o);
                eqb += __shfl_xor_sync(0xffffffffu, eqb, o);
            }
            if (on && part == 0) {
                const float ft2 = (float)(cx.base_total + cx.dtot[s]);
                cx.gy[s] = make_float2(ft2, 1.0f / ft2);
                cx.grow[s] = 4LL * (sm.sout_off[s] + item * p.out_stride);
                sm.m_sorted[lt + eqb] = (unsigned char)s;
                sm.m_lt[s] = (unsigned char)lt;
                sm.m_eq[s] = (unsigned char)eq;
            }
        }
        const int n_dense = sm.n_bern;
        if (ptid == 0) cx.n_dense = n_dense;
        bar_named(1, PC_HALF);
        // ---- job order.  The MAIN jobs (the window total of the median sparse slot: usually > 2/3 of the slots)
        // stream from PC_NBUF - PC_NOTH row buffers that never need a rebuild; the OTHER jobs (dense rows, minority
        // totals: each needs the builders) take turns in the remaining PC_NOTH buffers, so a rebuild is hidden behind
        // the main jobs' bulk copies instead of stalling the store thread.  Position p uses buffer (gj0 + p) mod PC_NBUF.
        int M = 0, R0 = S;
        if (S > n_dense) {
            const int smid = sm.m_sorted[n_dense + (S - n_dense) / 2];
            M = sm.m_eq[smid]; R0 = sm.m_lt[smid];
        }
        const int O = S - M, a = gj0 % PC_NBUF;
        // (the first round of buffers is all main: the main row is the cheapest to have ready at the start of a sequence)
        auto lane_type = [&](int q) { return (a + q) % PC_NBUF >= PC_NBUF - PC_NOTH; };
        auto other_type = [&](int q) { return q >= PC_NBUF && lane_type(q); };
        auto lanes_before = [&](int q) {
            int f = (q / PC_NBUF) * PC_NOTH;
            for (int r = q - q % PC_NBUF; r < q; ++r) f += lane_type(r) ? 1 : 0;
            return f;
        };
        auto others_before = [&](int q) { return q <= PC_NBUF ? 0 : lanes_before(q) - lanes_before(PC_NBUF); };   // other-type positions in [0, q)
        if (ptid < 64) {
            const int q = ptid;
            const int f = others_before(q);
            const bool exh = q < S && (other_type(q) ? f >= O : q - f >= M);
            const unsigned bal = __ballot_sync(0xffffffffu, exh);
            if (lane == 0) sm.m_exh[ptid >> 5] = bal;
        }
        bar_named(1, PC_HALF);
        if (ptid < S) {
            const int q = ptid;
            const unsigned b0 = sm.m_exh[0], b1 = sm.m_exh[1];
            const int E = b0 ? __ffs(b0) - 1 : (b1 ? 32 + __ffs(b1) - 1 : S);   // first position whose list is exhausted
            int rank;
            if (q < E) {
                const int f = others_before(q);
                if (other_type(q)) rank = f < R0 ? f : f + M;          // other index f -> sorted rank
                else rank = R0 + (q - f);                              // main index q - f
            } else {
                const int fE = others_before(E);
                if (other_type(E)) rank = R0 + (E - fE) + (q - E);     // the others ran out: the rest are main jobs
                else { const int o = fE + (q - E); rank = o < R0 ? o : o + M; }
            }
            cx.job_slot[q] = sm.m_sorted[rank];
        }
        bar_named(1, PC_HALF);
        if (ptid < S) {
            const int j = ptid, s = cx.job_slot[j];
            const int nb = (j < PC_NBUF || sm.kind_class[s] == 2 || job_key(cx.job_slot[j - PC_NBUF]) != job_key(s)) ? 1 : 0;
            cx.job_build[j] = (unsigned char)nb;
            cx.job_dst[j] = (unsigned long long)cx.grow[s] | (unsigned long long)nb;
        }
        if (!cx.defer) gj0 += S;
        cur_item = nx_item; cur_seq = nx_seq; cur_c0 = nx_c0; cur_L = nx_L; cur_phase = nx_phase; cur_m0 = nx_m0; cur_m1 = nx_m1;
        bar_named(1, PC_HALF);
        if (ptid == 0) mbar_arrive(&sm.ctx_full[b]);   // release: hand the context over to the consumers
    }
}

// the 4 finished output floats of one granule whose bins hold the exact float counts c01 / c23
template <bool STD>
__device__ __forceinline__ float4 finish_granule2(float2 c01, float2 c23, float2 fy, const Stats2& st) {
    const float2 yy = make_float2(fy.y, fy.y), nt = make_float2(-fy.x, -fy.x);
    float2 q01 = __fmul2_rn(c01, yy), q23 = __fmul2_rn(c23, yy);
    const float2 r01 = __ffma2_rn(q01, nt, c01), r23 = __ffma2_rn(q23, nt, c23);
    q01 = __ffma2_rn(r01, yy, q01); q23 = __ffma2_rn(r23, yy, q23);             // RN(count / total)
    if (STD) {
        const float2 d01 = __fadd2_rn(q01, st.nm01), d23 = __fadd2_rn(q23, st.nm23);
        const float2 t01 = __fmul2_rn(d01, st.rs01), t23 = __fmul2_rn(d23, st.rs23);
        const float2 e01 = __ffma2_rn(t01, st.ns01, d01), e23 = __ffma2_rn(t23, st.ns23, d23);
        q01 = __ffma2_rn(e01, st.rs01, t01); q23 = __ffma2_rn(e23, st.rs23, t23);   // RN((q - mean) / scale)
    }
    return make_float4(q01.x, q01.y, q23.x, q23.y);
}
__device__ __forceinline__ void cvt_granule(uint2 pk, float magic, float2& c01, float2& c23) {
    const float2 nmag = make_float2(-magic, -magic);
    c01 = make_float2(__uint_as_float(__byte_perm(pk.x, 0x4B000000u, 0x7410)), __uint_as_float(__byte_perm(pk.x, 0x4B000000u, 0x7432)));
    c23 = make_float2(__uint_as_float(__byte_perm(pk.y, 0x4B000000u, 0x7410)), __uint_as_float(__byte_perm(pk.y, 0x4B000000u, 0x7432)));
    c01 = __fadd2_rn(c01, nmag); c23 = __fadd2_rn(c23, nmag);                    // exact count + pseudocount
}

// RN(1/x) from the hardware approximation and the per-bin ulp correction computed in the kernel prologue
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_exact(float x, int corr) { return __int_as_float(__float_as_int(rcp_approx(x)) + corr); }

// scaler statistics of one granule from shared memory, ready for the packed ops
template <bool STD>
__device__ __forceinline__ Stats2 smem_stats2(const PcSmem& sm, int vec) {
    Stats2 s;
    s.nm01 = s.nm23 = make_float2(0.f, 0.f);
    s.ns01 = s.ns23 = make_float2(-1.f, -1.f);
    s.rs01 = s.rs23 = make_float2(1.f, 1.f);
    if (STD) {
        const float4 m = reinterpret_cast<const float4*>(sm.smean)[vec];
        const float4 sc = reinterpret_cast<const float4*>(sm.sscale)[vec];
        const char4 rc = reinterpret_cast<const char4*>(sm.srcorr)[vec];
        const float4 rs = make_float4(rcp_exact(sc.x, rc.x), rcp_exact(sc.y, rc.y), rcp_exact(sc.z, rc.z), rcp_exact(sc.w, rc.w));
        s.nm01 = make_float2(-m.x, -m.y); s.nm23 = make_float2(-m.z, -m.w);
        s.ns01 = make_float2(-sc.x, -sc.y); s.ns23 = make_float2(-sc.z, -sc.w);
        s.rs01 = make_float2(rs.x, rs.y); s.rs23 = make_float2(rs.z, rs.w);
    }
    return s;
}

// BUILDERS (warps 0..7): finished rows into the ring of row buffers
template <int OUT>
__device__ __forceinline__ void pc_builder(PcSmem& sm, const ProfParams& p) {
    constexpr int NB = PC_NBLD, GPT = PC_VEC / NB;   // granules per thread
    constexpr bool STD = OUT == IDL_OUT_STD_F32;
    const int tid = threadIdx.x;
    const float magic = 8388608.0f - (float)p.pseudocount;
    int gj0 = 0;                                     // jobs of the previous sequences (CTA lifetime)
    for (int it = 0;; ++it) {
        const int b = it & 1;
        mbar_wait(&sm.ctx_full[b], (it >> 1) & 1);
        PcCtx& cx = sm.ctx[b];
        const long long item = cx.item;
        if (item < 0) return;
        if (!cx.defer) {
            const int S = p.S;
            uint2 ck[GPT];
            float2 c01[GPT], c23[GPT];               // exact float counts (+ pseudocount) of this thread's bins
#pragma unroll
            for (int j = 0; j < GPT; ++j) {
                ck[j] = cx.clean16[tid + j * NB];
                cvt_granule(ck[j], magic, c01[j], c23[j]);
            }
            // all Bernoulli deltas of the sequence (TMA-loaded from the prepared buffer) into the per-ordinal scratch arrays in ONE scan
            const int n_delta = cx.n_delta;
            if (cx.n_dense > 0) {
                bar_named(2, NB);                    // every builder is done with the previous sequence's dense rows (own-bin resets)
                if (n_delta > 0) {
                    mbar_wait(&sm.delta_full[b], (uint32_t)cx.delta_phase);
                    const uint16_t* dl = sm.delta[b];
                    for (int r = tid; r < n_delta; r += NB) {
                        const uint32_t e = dl[r];
                        upd16(sm.dscratch[(e >> 12) & 3u], e & 0xFFFu, (e & 0x8000u) ? 1 : -1);
                    }
                }
                bar_named(2, NB);
            }
            unsigned key_cur = 0u;                   // window total (float bits) the register row val[] holds; 0: none
            float4 val[GPT];
#pragma unroll
            for (int g = 0; g < GPT; ++g) val[g] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = 0; j < S; ++j) {
                const int buf = (gj0 + j) % PC_NBUF, use = (gj0 + j) / PC_NBUF;
                if (!cx.job_build[j]) continue;
                const int s = cx.job_slot[j];
                const float2 fy = cx.gy[s];
                const bool dense = sm.kind_class[s] == 2;
                // The row's values are computed BEFORE the buffer is free (only the stores sit on the buffer's critical
                // path) and kept in registers: consecutive rebuilds with the same window total cost four stores per thread.
                const unsigned key_j = dense ? 0u : __float_as_uint(fy.x);
                if (dense || key_j != key_cur) {
                    key_cur = key_j;
#pragma unroll
                    for (int g = 0; g < GPT; ++g) {
                        const int vec = tid + g * NB;
                        float2 d01 = c01[g], d23 = c23[g];
                        if (dense) {   // own bins = clean + delta; the scratch is reset on the way
                            uint2* scr = reinterpret_cast<uint2*>(sm.dscratch[sm.bern_ord[s]]);
                            const uint2 w = scr[vec];
                            scr[vec] = make_uint2(PC_BIAS2, PC_BIAS2);
                            cvt_granule(make_uint2(ck[g].x + w.x - PC_BIAS2, ck[g].y + w.y - PC_BIAS2), magic, d01, d23);
                        }
                        val[g] = finish_granule2<STD>(d01, d23, fy, smem_stats2<STD>(sm, vec));
                    }
                }
                // the bulk copy of the buffer's previous job has been read (counter = truth, the mbarrier is only the way to sleep)
                while (ld_acquire_smem(&sm.free_count[buf]) < use) mbar_try_once(&sm.row_free[buf], (use & 1) ^ 1);
                float4* row = reinterpret_cast<float4*>(sm.rowbuf[buf]);
#pragma unroll
                for (int g = 0; g < GPT; ++g) row[tid + g * NB] = val[g];
                fence_proxy_async_smem();              // generic-proxy writes -> visible to the TMA engine
                mbar_arrive(&sm.row_built[buf]);
            }
            gj0 += S;
        }
        mbar_arrive(&sm.ctx_empty[b]);
    }
}

// STORE thread (warp 15, lane 0): dispatches the items and writes each job's row with one TMA bulk copy
__device__ __forceinline__ void pc_store(PcSmem& sm, const ProfParams& p) {
    int gj = 0;
    // ---- dispatcher.  The atomic and the dependent loads of (sequence, length, first chunk) are two global
    // round trips; they are issued one iteration before their results are needed, and a stall here is absorbed
    // by the rows the other roles have already finished.
    const int4* prep_meta = reinterpret_cast<const int4*>(reinterpret_cast<const unsigned char*>(p.prep) + prep_meta_off());
    auto load_info = [&](long long item, long long& seq, long long& c0, int& L, int4& m0, int4& m1) {
        seq = item; c0 = 0; L = 0;
        m0 = make_int4(0, 0, 0, 1); m1 = make_int4(0, 0, 0, 0);
        if (item < p.n_items) {
            if (p.sidx) seq = (long long)p.sidx[item];
            L = p.len[seq];
            c0 = p.chunk_off[seq];
            m0 = prep_meta[item * 2]; m1 = prep_meta[item * 2 + 1];
        }
    };
    auto publish = [&](int idx, long long item, long long seq, long long c0, int L, int4 m0, int4 m1) {
        const int qs = idx & (PC_QRING - 1);
        sm.q_item[qs] = item; sm.q_seq[qs] = seq; sm.q_c0[qs] = c0; sm.q_len[qs] = L; sm.q_meta0[qs] = m0; sm.q_meta1[qs] = m1;
        st_release_smem(&sm.q_head, idx + 1);
    };
    {
        long long it4[4], sq4[4], c4[4];
        int l4[4];
        int4 ma4[4], mb4[4];
        for (int i = 0; i < 4; ++i) it4[i] = (long long)atomicAdd(p.work_counter, 1ull);
        for (int i = 0; i < 4; ++i) load_info(it4[i], sq4[i], c4[i], l4[i], ma4[i], mb4[i]);
        for (int i = 0; i < 4; ++i) publish(i, it4[i], sq4[i], c4[i], l4[i], ma4[i], mb4[i]);
    }
    long long a_item = (long long)atomicAdd(p.work_counter, 1ull);   // index 4
    long long b_item = 0, b_seq = 0, b_c0 = 0;
    int b_L = 0;
    int4 b_m0 = make_int4(0, 0, 0, 1), b_m1 = make_int4(0, 0, 0, 0);
    for (int it = 0;; ++it) {
        const int b = it & 1;
        if (it >= 1) publish(it + 3, b_item, b_seq, b_c0, b_L, b_m0, b_m1);      // loaded during the previous iteration
        b_item = a_item;
        load_info(b_item, b_seq, b_c0, b_L, b_m0, b_m1);              // index it + 4
        a_item = (long long)atomicAdd(p.work_counter, 1ull);          // index it + 5
        mbar_wait(&sm.ctx_full[b], (it >> 1) & 1);
        PcCtx& cx = sm.ctx[b];
        const long long item = cx.item;
        if (item < 0) break;
        if (!cx.defer) {
            const int S = p.S;
            unsigned long long jd_next = cx.job_dst[0];
            for (int j = 0; j < S; ++j, ++gj) {
                const unsigned long long jd = jd_next;
                if (j + 1 < S) jd_next = cx.job_dst[j + 1];
                const int buf = gj % PC_NBUF;
                mbar_wait(&sm.row_full[buf], (gj / PC_NBUF) & 1);
                unsigned char* dst = reinterpret_cast<unsigned char*>(p.out) + (jd & ~15ull);
                bulk_store(dst, sm.rowbuf[buf], PC_F * 4);
                bulk_commit();
                if (gj >= PC_INFL) {
                    bulk_wait_read<PC_INFL>();         // all but the PC_INFL most recent copies have left shared memory
                    st_release_smem(&sm.free_count[(gj - PC_INFL) % PC_NBUF], (gj - PC_INFL) / PC_NBUF + 1);
                    mbar_arrive(&sm.row_free[(gj - PC_INFL) % PC_NBUF]);
                }
            }
        }
        mbar_arrive(&sm.ctx_empty[b]);
    }
    bulk_wait_read<0>();
    bulk_wait<0>();
}

// FIX warps (warps 8 .. 8+PC_NBUF-1, one per row buffer): make the buffer's row the job's row.  Subtract the
// job's removals into the warp's scratch (shared atomics on biased uint8 fields), claim each touched scratch
// word with atomicExch (the first visitor owns its four bins and resets it — duplicate k-mers in the removal
// list are harmless); once the buffer's previous bulk copy has been read, put the template value back into the
// bins the previous job changed (unless the builders rebuilt the row) and write this job's changed bins.
template <int OUT>
__device__ __forceinline__ void pc_fix(PcSmem& sm, const ProfParams& p) {
    constexpr int K = PC_K;
    constexpr bool STD = OUT == IDL_OUT_STD_F32;
    constexpr int RPL = 4;                             // removal entries per lane (<= 127 removals per job, host-checked)
    const int ftid = threadIdx.x - PC_NBLD, fw = ftid >> 5, lane = ftid & 31;
    if (fw >= PC_NBUF) {                               // spare warps: only the context hand-shake
        for (int it = 0;; ++it) {
            const int b = it & 1;
            mbar_wait(&sm.ctx_full[b], (it >> 1) & 1);
            if (sm.ctx[b].item < 0) return;
            mbar_arrive(&sm.ctx_empty[b]);
        }
    }
    uint32_t* scr = sm.sscratch + fw * PC_SCRW;
    float* row = sm.rowbuf[fw];
    int gj0 = 0, n_built = 0;                          // CTA lifetime: jobs of the previous sequences, rebuilds of this buffer
    uint32_t km_prev[RPL];                             // the bins the previous job of this buffer changed (0xFFFF: none) ...
    float vt_prev[RPL];                                // ... and the template values it found there
#pragma unroll
    for (int u = 0; u < RPL; ++u) { km_prev[u] = 0xFFFFu; vt_prev[u] = 0.f; }
    for (int it = 0;; ++it) {
        const int b = it & 1;
        mbar_wait(&sm.ctx_full[b], (it >> 1) & 1);
        PcCtx& cx = sm.ctx[b];
        const long long item = cx.item;
        if (item < 0) return;
        if (!cx.defer) {
            const int S = p.S;
            const uint16_t* clean_h = reinterpret_cast<const uint16_t*>(cx.clean16);
            // output value of one bin whose clean count changes by d (every lane owns exactly its own entries, so the
            // RPL evaluations of a lane are independent and the warp does not diverge)
            auto value = [&](uint32_t bin, int d, float2 fy) -> float {
                float q = div_rn((float)((int)clean_h[bin] + d + p.pseudocount), fy.x, fy.y);
                if (STD) { const float sc = sm.sscale[bin]; q = div_rn(q - sm.smean[bin], sc, rcp_exact(sc, sm.srcorr[bin])); }
                return q;
            };
            int j = (fw - gj0 % PC_NBUF + PC_NBUF) % PC_NBUF;      // first job of this sequence that lands in this buffer
            for (; j < S; j += PC_NBUF) {
                const int use = (gj0 + j) / PC_NBUF;
                const int s = cx.job_slot[j];
                const int n = sm.nbp[s] * K;           // 0 for clean and dense slots
                const uint16_t* rl = cx.rem + sm.rem_off[s] * K;
                const float2 fy = cx.gy[s];
                const bool rebuilt = cx.job_build[j] != 0;
                uint32_t km[RPL];
                float vnew[RPL];
#pragma unroll
                for (int u = 0; u < RPL; ++u) { km[u] = 0xFFFFu; vnew[u] = 0.f; }
                if (n > 0) {                           // (warp-uniform) nothing to prepare for clean and dense slots
                    int d[RPL];
#pragma unroll
                    for (int u = 0; u < RPL; ++u) {
                        const int r = lane + 32 * u;
                        km[u] = r < n ? (uint32_t)rl[r] : 0xFFFFu;
                    }
                    // multiplicity of each removed k-mer within this job: subtract into the scratch, read back, reset
#pragma unroll
                    for (int u = 0; u < RPL; ++u)
                        if (km[u] != 0xFFFFu) atomicSub(scr + (km[u] >> 2), 1u << ((km[u] & 3u) * 8u));
                    __syncwarp();
#pragma unroll
                    for (int u = 0; u < RPL; ++u)
                        d[u] = km[u] != 0xFFFFu ? (int)((scr[km[u] >> 2] >> ((km[u] & 3u) * 8u)) & 0xFFu) - 0x80 : 0;
                    __syncwarp();
#pragma unroll
                    for (int u = 0; u < RPL; ++u)
                        if (km[u] != 0xFFFFu) scr[km[u] >> 2] = PC_BIAS4;
#pragma unroll
                    for (int u = 0; u < RPL; ++u)
                        if (km[u] != 0xFFFFu) vnew[u] = value(km[u], d[u], fy);
                }
                if (rebuilt) {
                    mbar_wait(&sm.row_built[fw], n_built & 1);     // the builders wrote a fresh row (they waited for row_free)
                    ++n_built;
                } else {
                    mbar_wait(&sm.row_free[fw], (use & 1) ^ 1);    // the bulk copy of the buffer's previous job has been read
                    // same window total as the buffer's previous job: put the template values back where that job changed them
#pragma unroll
                    for (int u = 0; u < RPL; ++u)
                        if (km_prev[u] != 0xFFFFu) row[km_prev[u]] = vt_prev[u];
                    __syncwarp();
                }
                // the row now holds the template: remember its values at this job's bins (the next job's undo list), then overwrite
#pragma unroll
                for (int u = 0; u < RPL; ++u) {
                    km_prev[u] = km[u];
                    if (km[u] != 0xFFFFu) vt_prev[u] = row[km[u]];
                }
                __syncwarp();
#pragma unroll
                for (int u = 0; u < RPL; ++u)
                    if (km[u] != 0xFFFFu) row[km[u]] = vnew[u];
                fence_proxy_async_smem();              // generic-proxy writes -> visible to the TMA engine
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.row_full[fw]);
            }
            gj0 += S;
        }
        mbar_arrive(&sm.ctx_empty[b]);
    }
}

template <int OUT>
__global__ void __launch_bounds__(PC_NT, 1) profiles_pc_kernel(const ProfParams p, const __grid_constant__ Plan plan) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PcSmem& sm = *reinterpret_cast<PcSmem*>(smem_raw);
    const int tid = threadIdx.x;
    if (tid == 0) {
        sm.params = p; sm.rcorr_bad = 0;
        // the prepared buffer must have been written for exactly this call's items / variants / seed
        const PrepHeader* h = reinterpret_cast<const PrepHeader*>(p.prep);
        sm.prep_bad = (h->stamp != p.prep_stamp || h->n_items != p.n_items) ? 1 : 0;
    }
    __syncthreads();
    // launch-uniform slot tables (the host only takes this kernel with an inline plan: n_vars, S <= PC_MAXS)
    for (int i = tid; i < p.n_vars; i += PC_NT) sm.svars[i] = plan.vars[i];
    for (int i = tid; i < p.S; i += PC_NT) sm.sout_off[i] = plan.out_off[i];
    if (OUT == IDL_OUT_STD_F32)
        for (int i = tid; i < PC_F; i += PC_NT) {
            const float sc = p.scale[i];
            const int corr = __float_as_int(p.rscale[i]) - __float_as_int(rcp_approx(sc));
            sm.smean[i] = p.mean[i]; sm.sscale[i] = sc; sm.srcorr[i] = (signed char)corr;
            if (corr < -64 || corr > 64) sm.rcorr_bad = 1;
        }
    for (int i = tid; i < PC_DENSE * PC_PRIVW; i += PC_NT) (&sm.dscratch[0][0])[i] = PC_BIAS2;
    for (int i = tid; i < PC_NBUF * PC_SCRW; i += PC_NT) sm.sscratch[i] = PC_BIAS4;
    __syncthreads();
    if (tid == 0) {
        int ent = 0, nb = 0;
        for (int s = 0; s < p.S; ++s) {
            const VarDesc vd = sm.svars[s];
            int kc = 0;
            if (vd.kind == KIND_RANDOM_N) kc = vd.n_bp > 0 ? 1 : 0;
            else if (vd.kind != KIND_CLEAN) kc = 2;
            sm.kind_class[s] = kc;
            sm.nbp[s] = kc == 1 ? vd.n_bp : 0;
            sm.rem_off[s] = ent;
            sm.bern_ord[s] = kc == 2 ? nb : 0;
            if (kc == 1) ent += vd.n_bp;
            if (kc == 2) { sm.bern_slot[nb] = s; ++nb; }
        }
        sm.n_ent = ent;
        sm.n_bern = nb;
        sm.q_head = 0;
        for (int i = 0; i < 2; ++i) { mbar_init(&sm.seq_full[i], 1); mbar_init(&sm.delta_full[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&sm.ctx_full[i], 1); mbar_init(&sm.ctx_empty[i], PC_NBLD + PC_NFIX + 1); }
        for (int i = 0; i < PC_NBUF; ++i) { mbar_init(&sm.row_free[i], 1); mbar_init(&sm.row_built[i], PC_NBLD); mbar_init(&sm.row_full[i], 1); sm.free_count[i] = 0; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid >= PC_HALF) pc_producer<OUT>(sm);
    else if (tid < PC_NBLD) pc_builder<OUT>(sm, p);
    else if (tid < PC_NBLD + PC_NFIX) pc_fix<OUT>(sm, p);
    else if (tid == PC_NBLD + PC_NFIX) pc_store(sm, p);
}

}  // namespace idl
static_assert(sizeof(idl::PcSmem) <= 232448, "PcSmem exceeds the 227 KB dynamic shared memory limit");
