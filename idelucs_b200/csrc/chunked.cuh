// idelucs_b200 — chunked featurisation of LONG sequences (k = 6; BASELINE configs[4]: Fungi-shaped genomes, SURVEY §8e).
//
// The generic kernel gives a sequence to ONE CTA; a set whose lengths span 20 kb .. 2 Mb then serialises on a few CTAs.
// Here the long items (more than CH_MIN_LEN bases) are cut into tiles of CH_TILE_BLOCKS x 64 bases, the tiles of all long
// items form one list, and every CTA of a persistent grid takes an equal contiguous share of it:
//
//   plan   (1 CTA)      tiles per item -> exclusive scan (tile_off), rank of every long item, totals
//   tiles  (grid CTAs)  per tile: window ends counted with the k-1 bases of context in front of the tile
//                       (idelucs/kmers.pyx:38-50 is local: a window only needs its own k bases), the Bernoulli / explicit
//                       ("dense") slots' edits of the tile (+ one 64-base block of context on each side) turned into +-1
//                       deltas of separate int32 delta histograms; the CTA keeps accumulating in shared memory while its
//                       tiles stay inside one item and writes ONE partial (clean + delta histograms) per (CTA, item) —
//                       partial slot = rank(item) + CTA index, which is injective because both only grow along the list
//   reduce (1 CTA/item) sums the item's partials in CTA order (integers: exact, no global atomics), adds the delta
//                       histogram of a dense slot / applies a Random_N slot's removals to the summed histogram, and emits
//                       every slot's row in the requested output kind with the same arithmetic as the other kernels.
//
// Mutations follow the same counter-based RNG as everywhere else, so a chunked item equals the generic kernel's result bit
// for bit (tests/test_gpu_parity_long.py compares both with the oracle).  Included by kernels.cu.
#pragma once

namespace idl {

constexpr int CH_NT = 512;
constexpr int CH_TILE_BLOCKS = 256;      // 16 384 bases per tile
constexpr int CH_MAX_DENSE = 7;          // dense (Bernoulli / explicit) slots per item
constexpr int CH_F = 4096;

struct ChHeader {                        // device-side plan (start of the scratch buffer)
    long long n_tiles;
    long long n_long;
    int overflow;                        // more long items than the scratch was sized for: the generic kernel takes them
    int pad;
};

struct ChParams {
    ProfParams p;
    ChHeader* hdr;
    long long* tile_off;                 // [n_items + 1]
    int* long_rank;                      // [n_items]: rank among the long items (-1: short)
    int* partials;                       // [(max_long + grid)][1 + nd_cap][CH_F]
    long long max_long;
    int nd_cap;                          // delta histograms per partial
    int grid_tiles;                      // CTAs of the tile kernel
};

__device__ __forceinline__ bool ch_is_dense(int kind) {
    return kind == KIND_TRANSITION || kind == KIND_TRANSVERSION || kind == KIND_BOTH || kind == KIND_EXPLICIT;
}

// ---- plan ----
__global__ void __launch_bounds__(1024) ch_plan_kernel(const ChParams cp) {
    __shared__ long long s_tiles[32];
    __shared__ int s_long[32];
    __shared__ long long run_tiles;
    __shared__ int run_long;
    const ProfParams& p = cp.p;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) { run_tiles = 0; run_long = 0; }
    __syncthreads();
    for (long long base = 0; base < p.n_items; base += 1024) {
        const long long w = base + tid;
        int tiles = 0, is_long = 0;
        if (w < p.n_items) {
            const long long seq = p.sidx ? (long long)p.sidx[w] : w;
            const int L = p.len[seq];
            if (L >= CH_MIN_LEN) {
                const int nblocks = (L + RNG_BLOCK - 1) / RNG_BLOCK;
                tiles = (nblocks + CH_TILE_BLOCKS - 1) / CH_TILE_BLOCKS;
                is_long = 1;
            }
        }
        long long it = tiles;
        int il = is_long;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long a = __shfl_up_sync(0xffffffffu, it, o);
            const int b = __shfl_up_sync(0xffffffffu, il, o);
            if (lane >= o) { it += a; il += b; }
        }
        if (lane == 31) { s_tiles[wid] = it; s_long[wid] = il; }
        __syncthreads();
        long long wt = 0;
        int wl = 0;
        for (int g = 0; g < wid; ++g) { wt += s_tiles[g]; wl += s_long[g]; }
        const long long rt = run_tiles;
        const int rl = run_long;
        if (w < p.n_items) {
            cp.tile_off[w] = rt + wt + it - tiles;
            cp.long_rank[w] = is_long ? rl + wl + il - 1 : -1;
        }
        __syncthreads();
        if (tid == 1023) { run_tiles = rt + wt + it; run_long = rl + wl + il; }
        __syncthreads();
    }
    if (tid == 0) {
        cp.tile_off[p.n_items] = run_tiles;
        cp.hdr->n_tiles = run_tiles;
        cp.hdr->n_long = run_long;
        cp.hdr->overflow = run_long > cp.max_long ? 1 : 0;
        cp.hdr->pad = 0;
    }
}

// ---- tiles ----
struct ChSmem {
    alignas(16) uint32_t tcodes[(CH_TILE_BLOCKS + 2) * 4 + 8];   // the tile's packed bases incl. one context block on each side ...
    alignas(16) uint32_t tmask[(CH_TILE_BLOCKS + 2) * 2 + 8];    // ... and reset flags (window lookups of the edits hit shared memory)
    uint32_t list[LIST_CAP + 8];
    uint32_t gtabs[STABS][RNG_BLOCK];
    VarDesc svars[SVARS];
    int scan[CH_NT / 32 + 2];
    int seg_off[CH_MAX_DENSE + 1];
    int dense_var[CH_MAX_DENSE];         // variant index of the item's dense slots (slot order)
    int n_dense;
    alignas(16) int hist[1][CH_F];       // [1 + nd_cap][CH_F] (dynamic): clean counts, then one delta histogram per dense slot
};

template <int K>
__global__ void __launch_bounds__(CH_NT, 2) ch_tile_kernel(const ChParams cp, const __grid_constant__ Plan plan) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ChSmem& sm = *reinterpret_cast<ChSmem*>(smem_raw);
    const ProfParams& p = cp.p;
    const int tid = threadIdx.x, lane = tid & 31;
    const int nh = 1 + cp.nd_cap;
    if (cp.hdr->overflow) return;
    const long long T = cp.hdr->n_tiles, G = gridDim.x;
    const long long t_lo = (long long)blockIdx.x * T / G, t_hi = (long long)(blockIdx.x + 1) * T / G;
    if (t_lo >= t_hi) return;
    const bool cached = p.inline_plan != 0;
    if (cached)
        for (int i = tid; i < p.n_vars; i += CH_NT) sm.svars[i] = plan.vars[i];
    for (int i = tid; i < STABS * RNG_BLOCK; i += CH_NT)
        (&sm.gtabs[0][0])[i] = i < p.n_tabs * RNG_BLOCK ? (cached ? (&plan.gtab[0][0])[i] : p.gtab[i]) : 0u;
    const VarDesc* __restrict__ vars = cached ? sm.svars : p.vars;
    auto table = [&](int t) -> const uint32_t* { return t < STABS ? sm.gtabs[t] : p.gtab + t * RNG_BLOCK; };
    int* hist = &sm.hist[0][0];
    for (int i = tid; i < nh * CH_F; i += CH_NT) hist[i] = 0;
    // first item of this CTA's range: largest w with tile_off[w] <= t_lo among the items that own tiles
    long long item;
    {
        long long lo = 0, hi = p.n_items;   // invariant: tile_off[lo] <= t_lo < tile_off[hi]
        while (hi - lo > 1) {
            const long long mid = (lo + hi) >> 1;
            if (cp.tile_off[mid] <= t_lo) lo = mid; else hi = mid;
        }
        item = lo;
    }
    __syncthreads();
    long long t = t_lo;
    while (t < t_hi) {
        // ---- the item that owns tile t (items without tiles are skipped) ----
        while (cp.tile_off[item + 1] <= t) ++item;
        const long long seq = p.sidx ? (long long)p.sidx[item] : item;
        const int L = p.len[seq];
        const long long c0 = p.chunk_off[seq];
        const uint32_t* gcodes = p.codes + c0 * 4;
        const uint32_t* gnmask = p.nmask + c0 * 2;
        const uint32_t seq_id = (uint32_t)(p.seq_id0 + seq);
        const int nblocks = (L + RNG_BLOCK - 1) / RNG_BLOCK;
        const long long t_item0 = cp.tile_off[item], t_item1 = cp.tile_off[item + 1];
        const long long t_end = t_item1 < t_hi ? t_item1 : t_hi;   // this CTA's tiles of the item: [t, t_end)
        if (tid == 0) {   // the item's dense slots, in slot order
            int nd = 0;
            for (int s = 0; s < p.S; ++s) {
                const int v = p.sel ? p.sel[item * p.S + s] : s;
                if (ch_is_dense(vars[v].kind) && nd < CH_MAX_DENSE) sm.dense_var[nd++] = v;
            }
            sm.n_dense = nd;
        }
        __syncthreads();
        const int nd = sm.n_dense;
        for (; t < t_end; ++t) {
            const int b0 = (int)(t - t_item0) * CH_TILE_BLOCKS;
            const int b1 = b0 + CH_TILE_BLOCKS < nblocks ? b0 + CH_TILE_BLOCKS : nblocks;
            // ---- stage the tile (+ one 64-base block of context on each side, + one slack word) ----
            const int sb0 = b0 > 0 ? b0 - 1 : 0, sb1 = b1 + 1 < nblocks ? b1 + 1 : nblocks;
            __syncthreads();   // the previous tile's lookups are done
            for (int i = tid; i < (sb1 - sb0) * 4 + 4; i += CH_NT) sm.tcodes[i] = __ldg(gcodes + sb0 * 4 + i);
            for (int i = tid; i < (sb1 - sb0) * 2 + 2; i += CH_NT) sm.tmask[i] = __ldg(gnmask + sb0 * 2 + i);
            __syncthreads();
            // absolute word indices keep working through these (only staged words are ever dereferenced)
            const uint32_t* codes = sm.tcodes - sb0 * 4;
            const uint32_t* nmask = sm.tmask - sb0 * 2;
            // ---- clean window ends of the tile (half-chunks 2 b0 .. 2 b1) ----
            for (int h = 2 * b0 + tid; h < 2 * b1; h += CH_NT) {
                const uint2 w = make_uint2(codes[2 * h], codes[2 * h + 1]);
                count_half<K>(codes, nmask, h, w.x, w.y, [&](uint32_t kmer) { atomicAdd(&hist[kmer], 1); });
            }
            // ---- dense slots: edits of the tile's blocks (+ context) -> +-1 deltas.  Bernoulli slots jointly: work item =
            // ---- (slot, block), rounds of CH_NT items, one list with a segment per slot; explicit lists stay in global memory ----
            int span = b1 - b0;
            for (int s0 = b0; s0 < b1 && nd > 0;) {
                const int s1 = s0 + span < b1 ? s0 + span : b1;
                const int g0 = s0 > 0 ? s0 - 1 : 0, g1 = s1 + 1 < nblocks ? s1 + 1 : nblocks;   // generated blocks
                const int nbt = g1 - g0;
                const int lo = s0 * RNG_BLOCK;
                const long long hi = (long long)s1 * RNG_BLOCK;
                int base = 0;
                bool over = false;
                const int W = nd * nbt;
                for (int w0 = 0; w0 < W; w0 += CH_NT) {   // uniform trip count (CTA scan inside)
                    const int w = w0 + tid;
                    int d = 0, b = -1;
                    BlockMasks m;
                    m.a = m.b = m.ch = 0;
                    if (w < W) {
                        d = w / nbt;
                        const VarDesc vd = vars[sm.dense_var[d]];
                        if (vd.kind != KIND_EXPLICIT) {
                            b = g0 + (w - d * nbt);
                            m = block_masks(vd.kind, p.seed, seq_id, (uint32_t)vd.rng_id, b, L, nmask, table(vd.tab1), vd.slope1, table(vd.tab2), vd.slope2);
                        }
                        if (w - d * nbt == 0) sm.seg_off[d] = -1;   // set below (first block of the slot)
                    }
                    int total;
                    const int off = block_exscan<CH_NT>(block_masks_count(m), sm.scan, &total);
                    if (base + total > LIST_CAP) { over = true; break; }   // uniform
                    if (w < W && w - d * nbt == 0) sm.seg_off[d] = base + off;
                    if (b >= 0) block_masks_write(m, b, codes, sm.list + base + off);
                    base += total;
                }
                if (over) { span = span > 1 ? span >> 1 : 1; __syncthreads(); continue; }   // fewer blocks at a time (three always fit)
                if (tid == 0) sm.seg_off[nd] = base;
                __syncthreads();
                for (int i = tid; i < base; i += CH_NT) {   // thread <-> edit of any Bernoulli slot
                    int d = 0;
                    while (i >= sm.seg_off[d + 1]) ++d;
                    const int so = sm.seg_off[d], n = sm.seg_off[d + 1] - so;
                    const int pos = (int)(sm.list[i] >> 3);
                    int* dh = hist + (1 + d) * CH_F;
                    if (pos >= lo && pos < hi) apply_entry<K>(codes, nmask, L, sm.list + so, n, i - so, [&](uint32_t kmer, int dd) { atomicAdd(&dh[kmer], dd); });
                }
                for (int d = 0; d < nd; ++d) {
                    const VarDesc vd = vars[sm.dense_var[d]];
                    if (vd.kind != KIND_EXPLICIT) continue;
                    int* dh = hist + (1 + d) * CH_F;
                    const long long li = (long long)vd.explicit_idx * p.n_seqs_total + seq;
                    const uint32_t* glist = p.edits + p.edit_off[li];
                    const int n = (int)(p.edit_off[li + 1] - p.edit_off[li]);
                    int a = 0, z = n;   // first entry with pos >= lo
                    while (a < z) { const int mid = (a + z) >> 1; if ((int)(glist[mid] >> 3) < lo) a = mid + 1; else z = mid; }
                    for (int i = a + tid; i < n && (long long)(glist[i] >> 3) < hi; i += CH_NT)
                        apply_entry<K>(codes, nmask, L, glist, n, i, [&](uint32_t kmer, int dd) { atomicAdd(&dh[kmer], dd); });
                }
                __syncthreads();   // the list is rewritten by the next span / tile
                s0 = s1;
            }
        }
        // ---- this CTA's partial of the item ----
        __syncthreads();
        {
            int4* dst = reinterpret_cast<int4*>(cp.partials + ((size_t)cp.long_rank[item] + blockIdx.x) * (size_t)nh * CH_F);
            int4* src = reinterpret_cast<int4*>(hist);
            for (int i = tid; i < nh * CH_F / 4; i += CH_NT) { dst[i] = src[i]; src[i] = make_int4(0, 0, 0, 0); }
        }
        __syncthreads();
    }
    (void)lane;
}

// ---- reduce + emit ----
struct ChRedSmem {
    alignas(16) int hist[CH_F];                      // clean histogram of the item, patched in place by Random_N slots
    uint32_t list[LIST_CAP + 8];
    uint32_t tmp[LIST_CAP / 2 + 8];
    VarDesc svars[SVARS];
    long long sout_off[SVARS];
    int scan[CH_NT / 32 + 2];
    int dtot;
    int nvalid;
    int dense_of_slot[SVARS];            // dense ordinal of a slot of the current item (-1: not dense); slots >= SVARS are recomputed
};

template <int K, int OUT>
__global__ void __launch_bounds__(CH_NT, 2) ch_reduce_kernel(const ChParams cp, const __grid_constant__ Plan plan) {
    constexpr int F = CH_F, VEC = F / 4, VPT = VEC / CH_NT;
    constexpr int ESZ = (OUT == IDL_OUT_FREQ_F64 || OUT == IDL_OUT_CANON_F64) ? 8 : 4;
    __shared__ ChRedSmem sm;
    const ProfParams& p = cp.p;
    const int tid = threadIdx.x, lane = tid & 31;
    if (cp.hdr->overflow) return;
    const int nh = 1 + cp.nd_cap;
    const long long T = cp.hdr->n_tiles, G = cp.grid_tiles;
    const bool cached = p.inline_plan != 0;
    if (cached) {
        for (int i = tid; i < p.n_vars; i += CH_NT) sm.svars[i] = plan.vars[i];
        for (int i = tid; i < p.S; i += CH_NT) sm.sout_off[i] = plan.out_off[i];
    }
    const VarDesc* __restrict__ vars = cached ? sm.svars : p.vars;
    const long long* __restrict__ out_offs = cached ? sm.sout_off : reinterpret_cast<const long long*>(p.out_off);
    auto cta_of_tile = [&](long long t) {   // the CTA whose range [c T / G, (c + 1) T / G) holds tile t
        long long c = t * G / T;
        while (c > 0 && c * T / G > t) --c;
        while ((c + 1) * T / G <= t) ++c;
        return c;
    };
    for (long long item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int rank = cp.long_rank[item];
        if (rank < 0) continue;   // uniform
        __syncthreads();
        const long long seq = p.sidx ? (long long)p.sidx[item] : item;
        const long long t0 = cp.tile_off[item], t1 = cp.tile_off[item + 1];
        const long long c_first = cta_of_tile(t0), c_last = cta_of_tile(t1 - 1);
        // with fewer tiles than CTAs some CTAs in between own no tile at all (and wrote no partial)
        auto has_part = [&](long long c) { return c * T / G < (c + 1) * T / G; };
        ItemCtx cx;
        cx.L = p.len[seq];
        const long long c0 = p.chunk_off[seq];
        cx.codes = p.codes + c0 * 4;
        cx.nmask = p.nmask + c0 * 2;
        cx.seq_id = (uint32_t)(p.seq_id0 + seq);
        cx.seed = p.seed;
        // ---- clean histogram = sum of the partials' first histograms, in CTA order ----
        int nv = 0;
#pragma unroll
        for (int vv = 0; vv < VPT; ++vv) {
            const int vec = tid + vv * CH_NT;
            int4 a = make_int4(0, 0, 0, 0);
            for (long long c = c_first; c <= c_last; ++c) {
                if (!has_part(c)) continue;
                const int4 b = reinterpret_cast<const int4*>(cp.partials + ((size_t)rank + c) * (size_t)nh * F)[vec];
                a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
            }
            reinterpret_cast<int4*>(sm.hist)[vec] = a;
            nv += a.x + a.y + a.z + a.w;
        }
        if (tid == 0) {
            sm.nvalid = 0;
            int nd = 0;
            for (int s = 0; s < p.S && s < SVARS; ++s) {
                const int v = p.sel ? p.sel[item * p.S + s] : s;
                sm.dense_of_slot[s] = (ch_is_dense(vars[v].kind) && nd < CH_MAX_DENSE) ? nd++ : -1;
            }
        }
        __syncthreads();
        nv = warp_sum(nv);
        if (lane == 0 && nv) atomicAdd(&sm.nvalid, nv);
        __syncthreads();
        const int base_total = F * p.pseudocount + sm.nvalid;
        for (int s = 0; s < p.S; ++s) {
            const VarDesc vd = vars[p.sel ? p.sel[item * p.S + s] : s];
            int kind = (vd.kind == KIND_RANDOM_N && (vd.n_bp <= 0 || cx.L <= 0)) ? KIND_CLEAN : vd.kind;
            int dense = -1;
            if (ch_is_dense(kind)) {
                if (s < SVARS) dense = sm.dense_of_slot[s];
                else {   // (more slots than the table holds: recount the dense slots in front of s)
                    int nd = 0;
                    for (int q = 0; q < s; ++q) nd += ch_is_dense(vars[p.sel ? p.sel[item * p.S + q] : q].kind) ? 1 : 0;
                    dense = nd < CH_MAX_DENSE ? nd : -1;
                }
            }
            if (tid == 0) sm.dtot = 0;
            __syncthreads();
            if (kind == KIND_RANDOM_N) {   // removals applied to the summed histogram (and undone after the row is out)
                random_n_sorted<CH_NT>(cx, vd, sm.tmp, sm.list);
                int d = 0;
                for (int i = tid; i < vd.n_bp; i += CH_NT)
                    d += apply_entry<K>(cx.codes, cx.nmask, cx.L, sm.list, vd.n_bp, i, [&](uint32_t kmer, int dd) { atomicAdd(&sm.hist[kmer], dd); });
                d = warp_sum(d);
                if (lane == 0 && d) atomicAdd(&sm.dtot, d);
                __syncthreads();
            }
            // ---- the row: clean (+ delta histogram of a dense slot, summed over the partials) ----
            int4 row[VPT];
            int dsum = 0;
#pragma unroll
            for (int vv = 0; vv < VPT; ++vv) {
                const int vec = tid + vv * CH_NT;
                int4 a = reinterpret_cast<const int4*>(sm.hist)[vec];
                if (dense >= 0) {
                    for (long long c = c_first; c <= c_last; ++c) {
                        if (!has_part(c)) continue;
                        const int4 b = reinterpret_cast<const int4*>(cp.partials + (((size_t)rank + c) * (size_t)nh + 1 + dense) * F)[vec];
                        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
                        dsum += b.x + b.y + b.z + b.w;
                    }
                }
                row[vv] = a;
            }
            if (dense >= 0) {
                dsum = warp_sum(dsum);
                if (lane == 0 && dsum) atomicAdd(&sm.dtot, dsum);
                __syncthreads();
            }
            const int total = base_total + sm.dtot;
            const float ftot = (float)total;
            const float y = 1.0f / ftot;
            const bool big = total >= (1 << 24);
            void* out_row = reinterpret_cast<unsigned char*>(p.out) + (size_t)ESZ * (size_t)(out_offs[s] + item * p.out_stride);
            if constexpr (is_canon(OUT)) {
                // canonical rows pair bins of different threads: the row goes through sm.hist (whose counts wait in registers)
                int4 keep[VPT];
#pragma unroll
                for (int vv = 0; vv < VPT; ++vv) {
                    const int vec = tid + vv * CH_NT;
                    keep[vv] = reinterpret_cast<const int4*>(sm.hist)[vec];
                    reinterpret_cast<int4*>(sm.hist)[vec] = row[vv];
                }
                __syncthreads();
                emit_canon_row<K, CH_NT, OUT>(out_row, [&](uint32_t m) { return sm.hist[m] + p.pseudocount; }, p.mean, p.scale, sm.scan);
                __syncthreads();
#pragma unroll
                for (int vv = 0; vv < VPT; ++vv) reinterpret_cast<int4*>(sm.hist)[tid + vv * CH_NT] = keep[vv];
            } else {
#pragma unroll
            for (int vv = 0; vv < VPT; ++vv) {
                const int vec = tid + vv * CH_NT;
                const int4 h = row[vv];
                const int ci[4] = {h.x + p.pseudocount, h.y + p.pseudocount, h.z + p.pseudocount, h.w + p.pseudocount};
                const float cf[4] = {(float)ci[0], (float)ci[1], (float)ci[2], (float)ci[3]};
                float mean[4] = {0.f, 0.f, 0.f, 0.f}, scale[4] = {1.f, 1.f, 1.f, 1.f}, rscale[4] = {1.f, 1.f, 1.f, 1.f};
                if (OUT == IDL_OUT_STD_F32) {
                    const float4 m = reinterpret_cast<const float4*>(p.mean)[vec];
                    const float4 sc = reinterpret_cast<const float4*>(p.scale)[vec];
                    const float4 rs = reinterpret_cast<const float4*>(p.rscale)[vec];
                    mean[0] = m.x; mean[1] = m.y; mean[2] = m.z; mean[3] = m.w;
                    scale[0] = sc.x; scale[1] = sc.y; scale[2] = sc.z; scale[3] = sc.w;
                    rscale[0] = rs.x; rscale[1] = rs.y; rscale[2] = rs.z; rscale[3] = rs.w;
                }
                emit_granule<OUT>(out_row, vec, ci, cf, total, ftot, y, big, p.accumulate, mean, scale, rscale);
            }
            }
            __syncthreads();
            if (kind == KIND_RANDOM_N) {   // undo the removals
                for (int i = tid; i < vd.n_bp; i += CH_NT)
                    apply_entry<K>(cx.codes, cx.nmask, cx.L, sm.list, vd.n_bp, i, [&](uint32_t kmer, int dd) { atomicAdd(&sm.hist[kmer], -dd); });
                __syncthreads();
            }
        }
    }
}

}  // namespace idl
