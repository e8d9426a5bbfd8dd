/* idelucs_b200 — C ABI of the B200-native iDeLUCS featurisation / mimic / IIC-loss hot path.
 *
 * The reference (Kari-Genomics-Lab/iDeLUCS) has no FFI: its boundary for this path is a set
 * of Python callables.  Each entry point below names the reference interface it replaces
 * (file:line into the upstream repository); the Python shims in idelucs_b200/ keep the
 * reference names and signatures and bind these symbols through ctypes (INTEGRATION.md).
 *
 * Conventions
 *  - plain C, no C++ / torch types; every pointer whose name starts with d_ is a DEVICE
 *    pointer owned by the caller (e.g. the PyTorch caching allocator); the library never
 *    allocates or frees persistent device memory and never synchronises the stream;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it;
 *  - return value 0 = ok, otherwise an IDL_E* code; idl_last_error() gives the text
 *    (thread-local).  No exceptions, no exit();
 *  - packed sequence set ("seqset"):
 *      d_codes     uint32, 2 bits/base, 16 bases/word, big-endian inside the word
 *                  (A=0 C=1 G=2 T=3 — idelucs/kmers.pyx:19-34 numbering)
 *      d_nmask     uint32, 1 bit/base (bit 31-j of a word = base j): 1 = window reset
 *      d_chunk_off int64[n+1]: first 64-base chunk of every sequence (4 code words,
 *                  2 mask words per chunk); chunk_off[n] = number of chunks in use; the
 *                  buffers hold chunk_off[n]+1 chunks (one slack chunk)
 *      d_len       int32[n]: bases per sequence
 */
#ifndef IDELUCS_B200_H
#define IDELUCS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IDL_ABI_VERSION 3

enum {
    IDL_OK = 0,
    IDL_EINVAL = 1,      /* bad argument */
    IDL_ECUDA = 2,       /* CUDA runtime error (text in idl_last_error) */
    IDL_EUNSUPPORTED = 3 /* valid request this build cannot serve (e.g. k > 6) */
};

/* variant kinds: the transforms of idelucs/utils.py:54-135 */
enum {
    IDL_KIND_CLEAN = 0,        /* no mutation (kmersFasta(transform=None), utils.py:401) */
    IDL_KIND_TRANSITION = 1,   /* transition(p1), utils.py:54-76 */
    IDL_KIND_TRANSVERSION = 2, /* transversion(p2), utils.py:98-118 */
    IDL_KIND_BOTH = 3,         /* transition_transversion(p1, p2), utils.py:120-135 */
    IDL_KIND_RANDOM_N = 4,     /* Random_N(n_bp), utils.py:78-95 */
    IDL_KIND_EXPLICIT = 5      /* caller-supplied edit list (parity with the reference's own RNG) */
};

/* output kinds of idl_profiles */
enum {
    IDL_OUT_COUNTS_I32 = 0, /* raw window counts, no pseudocount (kmers.pyx:2-50) */
    IDL_OUT_FREQ_F32 = 1,   /* float32((count+pc)/sum)  (utils.py:242-250 then :353 astype) */
    IDL_OUT_STD_F32 = 2,    /* (freq32 - mean32) / scale32  (utils.py:358-366 via sklearn): IEEE float32 division (subnormal quotients
                             * included) when every scale32 is a finite, normal float, which idl_scaler_finalize guarantees for
                             * frequency columns.  A zero or infinite scale, or a subnormal one whose reciprocal overflows, gives
                             * NaN where IEEE division gives +-inf, 0 or a finite quotient */
    IDL_OUT_FREQ_F64 = 3,   /* float64 (count+pc)/sum  (utils.py:250) */
    /* canonical k-mer rows of kmersFasta(reduce=True) (utils.py:246-250): R = idl_revcomp_canonical(k) columns in its order;
     * each value is 8 + the matching frequency kind */
    IDL_OUT_CANON_F32 = 9,      /* float32 of IDL_OUT_CANON_F64's float64 quotient */
    IDL_OUT_CANON_STD_F32 = 10, /* (canon32 - mean32[r]) / scale32[r], IEEE float32 */
    IDL_OUT_CANON_F64 = 11      /* float64 f_r / T */
};

/* One mimic variant.  rng_id is the variant's identity in the counter-based RNG, so the
 * same (seed, sequence id, rng_id) always regenerates the same mimic, in any batch, on any
 * rank.  explicit_idx selects the edit list block for IDL_KIND_EXPLICIT. */
typedef struct idl_variant {
    int32_t kind;
    int32_t rng_id;
    int32_t n_bp;         /* Random_N */
    int32_t explicit_idx; /* EXPLICIT: lists are d_edit_off[explicit_idx * n_seqs_total + seq] */
    double p1;            /* transition probability */
    double p2;            /* transversion probability */
} idl_variant;

int idl_abi_version(void);
const char* idl_last_error(void);
/* number of CUDA kernels this library has launched in this process so far (bench.py reports the difference over its timed
 * region as gpu_launches; kernels replayed from a captured CUDA graph are not counted) */
long long idl_launch_count(void);

/* T[g-1] = floor((1-(1-p)^g) * 2^32), g = 1..64: the geometric gap table the rng mode
 * uses for an iid Bernoulli(p) process (host function; exported for the parity tests). */
int idl_geometric_table(double p, uint32_t* out64);

/* K1 — replaces check_sequence (idelucs/utils.py:26-51) + the byte LUT of kmer_counts
 * (idelucs/kmers.pyx:19-34).  d_ascii: concatenated sequence bytes; d_byte_off int64[n+1].
 * alphabet 0 = check_sequence mapping (acgtu -> ACGTT, IUPAC/'-' -> N, invalid bytes are
 * reported), 1 = strict kmers.pyx LUT (only 'A','C','G','T' are bases, nothing is invalid).
 * d_bad uint64[n] must be preset to 0xFF..FF by the caller; after the call an entry is
 * (pos << 3 | cls) of the first offending byte (cls 5 = whitespace that check_sequence
 * deletes, 6 = invalid byte) or still all-ones.  max_len = longest sequence (host hint). */
int idl_pack(const uint8_t* d_ascii, const int64_t* d_byte_off, int64_t n, int alphabet, int64_t max_len,
             const int64_t* d_chunk_off, uint32_t* d_codes, uint32_t* d_nmask, int32_t* d_len,
             unsigned long long* d_bad, void* stream);

/* workspace (bytes) idl_profiles needs in d_workspace */
size_t idl_profiles_workspace_bytes(void);

/* K2 + K3 — replaces kmer_counts (idelucs/kmers.pyx:2-50), the per-record body of
 * kmersFasta (idelucs/utils.py:239-250) and the mimic passes of AugmentFasta
 * (idelucs/utils.py:330-351).
 *
 * Work items: n_items; item w processes sequence d_sidx[w] (or w when d_sidx is NULL) and,
 * for s in [0, S): variant slot d_sel[w*S+s] (or s when d_sel is NULL; then S must equal
 * n_variants).  Row (s, w) of the output is written at element offset
 * out_off[s] + w*out_stride of d_out (elements of the out_kind's type; multiples of 4 and d_out 16-byte aligned: rows are
 * written as 16-byte vectors, IDL_EINVAL otherwise).
 * The RNG sequence id of an item is seq_id0 + its sequence index.
 * d_edit_off / d_edits: CSR edit lists for IDL_KIND_EXPLICIT variants (entry = pos<<3 | val,
 * val 0..3 = set A/C/G/T, 4 = set N; position-sorted and unique per list; positions < 2^29, which also bounds the length of
 * sequences that take a non-clean variant — clean counting accepts any length < 2^31), n_seqs_total =
 * number of sequences the CSR is indexed over.  d_mean/d_scale: float32[4^k] for
 * IDL_OUT_STD_F32.
 * Canonical kinds (IDL_OUT_CANON_*): row width R = idl_revcomp_canonical(k), column r = canonical k-mer m_r of that list.
 * With a = count[m_r] + pseudocount and b = count[revcomp(m_r)] + pseudocount, f_r = int((a + b) * 0.5) (a palindrome gives
 * a) and T = sum of the R values f_r (an exact integer, not the window total); CANON_F64 = f_r / T in float64, CANON_F32 =
 * float32 of that quotient, CANON_STD_F32 = (CANON_F32 - d_mean[r]) / d_scale[r] with d_mean / d_scale float32[R].  This is
 * idl_normalize_counts(idl_revcomp_fold(counts + pseudocount)) bit for bit, without the [n, 4^k] count rows.  Any out_off /
 * out_stride; idl_profiles_chunked takes them too, idl_profiles_prepared does not.  accumulate: bit 0 set (COUNTS only) adds into d_out like kmers.pyx does; bits 8..15 = n > 0 caps the generic
 * kernel at n CTAs per SM (a caller that overlaps the call with other work on another stream leaves room for it; 0 = fill the GPU).
 * d_status int32[n_items] (optional, zero on entry): scratch flags of the fast kernels (bit 1 marks items handed to the generic
 * kernel inside a call; clear again when the work is done).  No rate or length makes a mutation get dropped: edit lists that
 * do not fit on chip are generated in smaller tiles.
 * Nothing is cached between calls: descriptors, offsets and gap tables of calls with <= 64 variants / slots and <= 4 distinct
 * rates travel as kernel parameters (such calls enqueue no host->device copy and can be captured in a CUDA graph); bigger
 * plans are copied into d_workspace on `stream`. */
int idl_profiles(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                 const int32_t* d_len, int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items,
                 int64_t seq_id0, int k, const idl_variant* variants, int n_variants, const int32_t* d_sel,
                 int S, uint64_t seed, const int64_t* d_edit_off, const uint32_t* d_edits, int out_kind,
                 void* d_out, const int64_t* out_off, int64_t out_stride, int pseudocount, int accumulate,
                 const float* d_mean, const float* d_scale, int32_t* d_status, void* d_workspace,
                 size_t workspace_bytes, void* stream);

/* Column statistics of ONE variant's float32 frequency profiles without materialising them —
 * replaces the t_norm pass + StandardScaler.fit of AugmentFasta (idelucs/utils.py:330, 354-359):
 * every CTA accumulates shifted float64 column sums of the rows it produces and emits one
 * (count, mean, M2) part; feed d_partials / d_part_n / *n_parts to idl_scaler_finalize (after
 * all-gathering the parts of every rank when sharded).  d_partials double[max_parts][2][4^k],
 * d_part_n double[max_parts]; max_parts >= 8 x number of SMs.  Rows are assigned to CTAs statically, so the sums are
 * run-to-run identical.  Any k <= 6 and any variant kind (generic kernel); for the k = 6 schedule use idl_profiles_prepare,
 * which shares the mutation work with the profile pass. */
int idl_profile_stats(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off, const int32_t* d_len,
                      int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items, int64_t seq_id0, int k,
                      const idl_variant* variant, uint64_t seed, const int64_t* d_edit_off, const uint32_t* d_edits,
                      int pseudocount, double* d_partials, double* d_part_n, int max_parts, int* n_parts,
                      int32_t* d_status, void* d_workspace, size_t workspace_bytes, void* stream);

/* Whole-schedule featurisation in two calls (k = 6): AugmentFasta (idelucs/utils.py:321-368) needs the StandardScaler
 * statistics of pass 0 (t_norm) before it can write any standardised row, so every sequence is visited twice.
 * idl_profiles_prepare visits it ONCE for everything the Bernoulli mimics need: it writes, into the caller-owned buffer
 * d_prep (idl_prepare_bytes(n_items) bytes, 16-byte aligned), the +-1 histogram deltas of every transition / transversion /
 * combined variant (at most 3) and the uint16 histogram + window total of variants[0] (clean or one of those), and — when
 * d_partials is given — the (count, mean, M2) parts of variants[0]'s float32 frequencies exactly like idl_profile_stats
 * (d_partials double[max_parts][2][4096], d_part_n double[max_parts], max_parts >= 8 x SMs, *n_parts on return).
 * idl_profiles_prepared is idl_profiles (float32 outputs, no selection, no explicit lists) for the SAME sequences, items,
 * variants, seed and pseudocount: its k = 6 producer/consumer kernel loads the prepared deltas instead of generating the
 * mutations again.  The buffer carries a stamp of what it was prepared for; on a mismatch (or for the few items the prepare
 * pass flags: longer than 20 480 bases, on-chip list overflows) the generic kernel computes the rows — results are identical
 * either way.  The stamp identifies the sequences and the items by address (d_codes, d_sidx), not by content: rewriting
 * the packed sequences or the item list in place between the two calls is not noticed.  d_status int32[n_items] must be
 * zero on entry of each call and is zero again afterwards. */
size_t idl_prepare_bytes(int64_t n_items);
int idl_profiles_prepare(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off, const int32_t* d_len,
                         int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items, int64_t seq_id0, int k,
                         const idl_variant* variants, int n_variants, uint64_t seed, int pseudocount, void* d_prep, size_t prep_bytes,
                         double* d_partials, double* d_part_n, int max_parts, int* n_parts, int32_t* d_status, void* d_workspace,
                         size_t workspace_bytes, void* stream);
int idl_profiles_prepared(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                          const int32_t* d_len, int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items,
                          int64_t seq_id0, int k, const idl_variant* variants, int n_variants, uint64_t seed, int out_kind,
                          void* d_out, const int64_t* out_off, int64_t out_stride, int pseudocount,
                          const float* d_mean, const float* d_scale, int32_t* d_status, const void* d_prep, size_t prep_bytes,
                          void* d_workspace, size_t workspace_bytes, void* stream);

/* idl_profiles for sets with LONG sequences (BASELINE configs[4]: Fungi-shaped genomes; the reference takes any length
 * < 2^31, idelucs/kmers.pyx:14-16).  Same arguments and results as idl_profiles; with k = 6 the items of >= 65 536 bases are
 * cut into 16 384-base tiles that the whole grid shares (window ends counted with k-1 bases of context, mutations of a tile
 * generated with one 64-base block of context on each side), per-(CTA, item) int32 partial histograms in d_scratch and an
 * exact second-stage reduction — no global atomics, no single CTA serialising a 2 Mb genome.  Shorter items (and other k)
 * take the generic kernel in the same call.  d_scratch: idl_profiles_chunked_bytes(n_items, max_long_items, variants,
 * n_variants, S) bytes, 16-byte aligned; max_long_items >= number of items with >= 65 536 bases (if the device finds
 * more, the generic kernel computes them: same results).  At most 7 Bernoulli / explicit slots per item (else: 0 bytes /
 * generic kernel). */
size_t idl_profiles_chunked_bytes(int64_t n_items, int64_t max_long_items, const idl_variant* variants, int n_variants, int S);
int idl_profiles_chunked(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                         const int32_t* d_len, int64_t n_seqs_total, const int32_t* d_sidx, int64_t n_items,
                         int64_t seq_id0, int k, const idl_variant* variants, int n_variants, const int32_t* d_sel,
                         int S, uint64_t seed, const int64_t* d_edit_off, const uint32_t* d_edits, int out_kind,
                         void* d_out, const int64_t* out_off, int64_t out_stride, int pseudocount, int accumulate,
                         const float* d_mean, const float* d_scale, void* d_scratch, size_t scratch_bytes, int64_t max_long_items,
                         void* d_workspace, size_t workspace_bytes, void* stream);

/* Convenience form of the above for kmer_counts (idelucs/kmers.pyx:2-50): raw int32 counts
 * of every sequence into d_counts[n, 4^k] (accumulating when accumulate != 0). */
int idl_kmer_counts(const uint32_t* d_codes, const uint32_t* d_nmask, const int64_t* d_chunk_off,
                    const int32_t* d_len, int64_t n, int k, int32_t* d_counts, int accumulate,
                    void* d_workspace, size_t workspace_bytes, void* stream);

/* K4 — replaces sklearn StandardScaler.fit as called at idelucs/utils.py:358-359 (float32
 * t_norm profiles) and :404-405 (float64 clean profiles).
 * idl_colstats: per-column (count, mean, M2) partials of a row-major [n, F] matrix
 * (is_f64: 0 = float32, 1 = float64) into d_partials double[n_parts][2][F] and
 * d_part_n double[n_parts]; n_parts = idl_colstats_parts(n).
 * idl_scaler_finalize: Chan-merges n_parts partials in index order (deterministic) and
 * emits float64 mean/var/scale with sklearn's near-constant rule (scale 1) plus float32
 * copies.  Multi-GPU: all-gather the partials of every rank and finalize over all of them. */
int idl_colstats_parts(int64_t n);
int idl_colstats(const void* d_x, int is_f64, int64_t n, int F, double* d_partials, double* d_part_n,
                 void* stream);
int idl_scaler_finalize(const double* d_partials, const double* d_part_n, int n_parts, int F, double* d_mean64,
                        double* d_var64, double* d_scale64, float* d_mean32, float* d_scale32, void* stream);

/* replaces StandardScaler.transform at idelucs/utils.py:361-363 (float32, in place or out of
 * place: (x - mean32) / scale32 with IEEE float32 rounding; any F >= 1, 128-bit accesses when
 * F % 4 == 0 and all four pointers are 16-byte aligned) and :405 (float64:
 * (x - mean64) / scale64, optionally also written as float32 like models.py:163 casts it). */
int idl_standardize_f32(const float* d_x, float* d_out, int64_t n, int F, const float* d_mean32,
                        const float* d_scale32, void* stream);
int idl_standardize_f64(const double* d_x, double* d_out64, float* d_out32, int64_t n, int F,
                        const double* d_mean64, const double* d_scale64, void* stream);

/* K6 — index maps of an int32 count matrix [n, 4^k] (SURVEY §8f rank 4).
 * idl_cgr_map: replaces cgr() (idelucs/kmers.pyx:53-123): d_cgr[row, (cgr_i << k) + cgr_j] (+)= d_counts[row, kmer] —
 *   the FCGR cell of every k-mer (same windows as kmer_counts; verified cgr[cgr_index(m)] == kmer_counts[m]).
 * idl_revcomp_canonical: the canonical k-mer list of kmer_rev_comp (idelucs/utils.py:208-221: kmer <= reverse
 *   complement, increasing) into a HOST array of >= 4^k ints (NULL: only count); returns its length R.
 * idl_revcomp_fold: replaces kmer_rev_comp on the integer count vector the reference applies it to
 *   (utils.py:246-247, 268-269): d_out[row, r] = int((c[kmer_r] + c[revcomp(kmer_r)]) * 0.5) — the reference's
 *   in-place float product is truncated back into its int32 array.
 * idl_normalize_counts: counts / np.sum(counts) (utils.py:250, 272) per row of an int32 [n, R] matrix, float64
 *   and / or float32(float64) output. */
int idl_cgr_map(const int32_t* d_counts, int64_t n, int k, int32_t* d_cgr, int accumulate, void* stream);
int idl_revcomp_canonical(int k, int32_t* h_index);
int idl_revcomp_fold(const int32_t* d_counts, int64_t n, int k, const int32_t* d_canon, int R, int32_t* d_out,
                     void* stream);
int idl_normalize_counts(const int32_t* d_counts, int64_t n, int R, double* d_out64, float* d_out32, void* stream);

/* K5 — replaces IID_loss / compute_joint (idelucs/LossFunctions.py:20-62), forward and
 * backward in one launch.  d_z1, d_z2: float32 [B, C] row-major.  Outputs (each optional,
 * NULL to skip): d_loss float32[1]; d_joint float32[C, C] (symmetrised, normalised,
 * unclamped — compute_joint's return value); d_dz1, d_dz2 float32 [B, C] = dLoss/dz.
 * C <= idl_iid_loss_max_clusters().  d_workspace: idl_iid_loss_workspace_bytes(C) bytes of
 * scratch (fixed-order partial sums; no float atomics, results are run-to-run identical).
 * C <= 16 (every configuration of Example/ALL_RESULTS.tsv): one ordinary CTA.  C > 16: S2 = S + S^T (S = z1^T z2) into
 * the workspace, the launches of idl_iid_joint_algebra on it, then dz1 = z2 dS and dz2 = z1 dS (the workspace holds S2, dS and
 * the algebra's scratch). */
int idl_iid_loss_max_clusters(void);
size_t idl_iid_loss_workspace_bytes(int C);
int idl_iid_loss(const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps, float* d_loss,
                 float* d_joint, float* d_dz1, float* d_dz2, void* d_workspace, size_t workspace_bytes,
                 void* stream);
/* the same with the caller's weighting folded in (idelucs/models.py:128: loss = (1 - w) info_nce + w IID_loss): the gradients are
 * multiplied by grad_scale and d_loss receives loss_weight * loss + add_weight * (*d_add) (d_add: a device float written earlier
 * on the same stream, e.g. the InfoNCE loss; NULL = nothing added) — the whole training loss and its gradients without
 * a single framework kernel between the two fused losses. */
int idl_iid_loss_scaled(const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps, float grad_scale, float loss_weight,
                        const float* d_add, float add_weight, float* d_loss, float* d_joint, float* d_dz1, float* d_dz2, void* d_workspace,
                        size_t workspace_bytes, void* stream);

/* The C x C part of the same loss for callers that issue its three contractions as library GEMMs (worth it for large C, e.g. the
 * 200 output units of the n_clusters = 0 path): d_S2 = S + S^T with S = z1^T z2, [C, C] row-major, on entry; outputs (each optional):
 * d_loss (weighted and combined like idl_iid_loss_scaled), d_joint [C, C], d_dS [C, C] = grad_scale * dLoss/dS_sym (symmetric), from
 * which dLoss/dz1 = z2 dS and dLoss/dz2 = z1 dS.  d_scratch: 6 C floats.  Four small launches, fixed-order reductions, any C. */
int idl_iid_joint_algebra(const float* d_S2, int C, float lamb, float eps, float grad_scale, float loss_weight, const float* d_add,
                          float add_weight, float* d_loss, float* d_joint, float* d_dS, float* d_scratch, void* stream);

/* F2 — replaces info_nce_loss (idelucs/LossFunctions.py:65-98; weight 1 - w = 0.75 of the training loss, models.py:128) on the
 * two views stacked as one [n2 = 2B, D] float32 matrix (rows 0..B-1 = first view).  The two dense contractions stay library GEMMs
 * issued by the caller (strict fp32): S = fn fn^T and d loss / d fn = W fn.  Around them:
 *   idl_nce_normalize           fn = F.normalize(h) (x / max(||x||, 1e-12)), d_inv_norm[n2] = the factors
 *   idl_nce_softmax_xent        d_sim [n2, n2] holds S on entry; the loss (self-masked log-softmax of S / temperature, cross-entropy
 *                               against the other view, mean over rows) goes to d_loss, and S is overwritten IN PLACE by
 *                               W = (P + P^T - 2 Y) / (n2 T) (zero diagonal); d_lse, d_rowloss: n2 floats of scratch each
 *   idl_nce_normalize_backward  dh = inv_norm (dfn - fn (fn . dfn)) per row
 * Fixed-order reductions: results are run-to-run identical. */
int idl_nce_normalize(const float* d_h, int n2, int D, float* d_fn, float* d_inv_norm, void* stream);
int idl_nce_softmax_xent(float* d_sim, int n2, float temperature, float* d_lse, float* d_rowloss, float* d_loss, void* stream);
/* the same with W multiplied by grad_scale (the weight 1 - w of this loss in idelucs/models.py:128), so that the gradient
 * leaves the kernels already weighted; d_loss still receives the unweighted loss */
int idl_nce_softmax_xent_scaled(float* d_sim, int n2, float temperature, float grad_scale, float* d_lse, float* d_rowloss, float* d_loss,
                                void* stream);
int idl_nce_normalize_backward(const float* d_dfn, const float* d_fn, const float* d_inv_norm, int n2, int D, float* d_dh, void* stream);
/* the same with dfn given as n_parts partial products [n_parts, n2, D] (the caller splits the W fn contraction over its inner
 * dimension into one batched GEMM — a [n2, n2] x [n2, D] product alone has too few output tiles to fill the GPU); the parts are
 * added in index order */
int idl_nce_normalize_backward_parts(const float* d_dfn_parts, int n_parts, const float* d_fn, const float* d_inv_norm, int n2, int D,
                                     float* d_dh, void* stream);

/* Global-batch loss of the data-parallel step: W = world ranks of b pairs each compute (1 - w) InfoNCE + w IIC of the B = W b pairs
 * together, the loss one GPU computes on the whole batch.  The global stacked batch is [true rows of rank 0 .. W-1 ; modified rows
 * of rank 0 .. W-1]: local row q of rank r (its own stacked [2b, .] batch) is global row r b + q for q < b, else B + r b + (q - b).
 * What a rank needs of the others is read through HOST arrays of `world` device addresses (entry r = rank r's buffer: symmetric
 * memory, or the slots of an all-gathered tensor), always summed in rank order, so every rank computes the same bits.  The caller
 * synchronises the ranks between writing a buffer and the peers' reads of it.
 *   idl_iid_partial_s2           d_S2 [C, C] = S + S^T with S = z1^T z2 over this rank's b pairs (fixed order, exactly symmetric)
 *   idl_iid_global_finish        S2 = sum of the ranks' partials; the IIC loss and this rank's dz1 = z2 dS, dz2 = z1 dS, weighted and
 *                                combined like idl_iid_loss_scaled.  C <= 16: one kernel; larger C: the sum into the workspace,
 *                                idl_iid_joint_algebra on it, one contraction kernel.  d_workspace: idl_iid_loss_workspace_bytes(C)
 *   idl_nce_gather_rows          d_fn_all [2B, D] in global row order from every rank's normalised latent fn [2b, D]
 *   idl_nce_softmax_xent_rows    d_sim [2b, 2B] = fn fn_all^T on entry (this rank's rows); overwritten IN PLACE by grad_scale G_r,
 *                                G = (P - Y) / (2B T) (P the self-masked softmax rows, Y the positive pairs, G + G^T = the W of
 *                                idl_nce_softmax_xent); d_rowloss[2b] = each row's cross-entropy
 *   idl_nce_normalize_backward_global  dh of this rank's rows: dfn = (sum of n_parts local parts [n_parts, 2b, D] of G_r fn_all) +
 *                                (row gi of sum over the ranks of G_r'^T fn_r'), then the normalisation's backward.  Every peer
 *                                buffer holds [2B, D] of G_r'^T fn_r' followed by that rank's 2b row losses; d_loss (optional)
 *                                receives their sum over 2B, the global InfoNCE loss.  D <= 128.
 * world <= 16; peer addresses 4-byte aligned. */
int idl_iid_partial_s2(const float* d_z1, const float* d_z2, int B, int C, float* d_S2, void* stream);
int idl_iid_global_finish(const uint64_t* h_s2_peers, int world, const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps,
                          float grad_scale, float loss_weight, const float* d_add, float add_weight, float* d_loss, float* d_dz1, float* d_dz2,
                          void* d_workspace, size_t workspace_bytes, void* stream);
int idl_nce_gather_rows(const uint64_t* h_fn_peers, int world, int b, int D, float* d_fn_all, void* stream);
int idl_nce_softmax_xent_rows(float* d_sim, int b, int rank, int world, float temperature, float grad_scale, float* d_rowloss, void* stream);
int idl_nce_normalize_backward_global(const float* d_dfn_parts, int n_parts, const uint64_t* h_prod_peers, int world, const float* d_fn,
                                      const float* d_inv_norm, int b, int D, int rank, float* d_dh, float* d_loss, void* stream);

/* ReLU + Dropout(p) of the encoder (idelucs/PytorchUtils.py:36-44) fused with the tail of the Linear before it, one pass each way.
 * forward: v = sum over the n_parts partial products d_parts[n_parts, M, N] (n_parts = 1: a plain activation matrix) + d_bias[N]
 * (NULL: none); d_out = (v > 0 and kept) ? v / (1 - p) : 0.  The keep decision of an element in training step *d_step (device
 * int64, NULL = 0; read at run time, so a CUDA graph replays the call with a fresh mask) is a Philox4x32-10 word keyed by seed, the
 * step, the element index and `tag` (one per layer).  backward: d_dx = d_out > 0 ? d_dy / (1 - p) : 0 — no mask is stored.
 * N a multiple of 4. */
int idl_relu_dropout_forward(const float* d_parts, int n_parts, const float* d_bias, int64_t M, int N, float p, uint64_t seed,
                             const int64_t* d_step, uint32_t tag, float* d_out, void* stream);
int idl_relu_dropout_backward(const float* d_out, const float* d_dy, int64_t n, float p, float* d_dx, void* stream);
/* the same tail without activation: d_out[M, N] = sum over d_parts[n_parts, M, N] + d_bias[N] (NULL: none) */
int idl_sum_parts_bias(const float* d_parts, int n_parts, const float* d_bias, int64_t M, int N, float* d_out, void* stream);

/* Row ids of the reference's x_train (idelucs/utils.py:321-389: row r = sequence r mod N paired with mimic r div N + 1) -> the
 * arguments of idl_profiles' selection mode for one batch: d_sidx[n] = sequence index, d_sel[n, 2] = (0, mimic slot).  Replaces the
 * index arithmetic AugmentedDataset.__getitem__ does per item. */
int idl_pair_selection(const int64_t* d_pair_ids, int n, int64_t n_seqs, int32_t* d_sidx, int32_t* d_sel, void* stream);

/* Optimiser step of the data-parallel consumer (idelucs/models.py:86 torch.optim.RMSprop(lr, weight_decay=0.01); momentum 0,
 * not centred) on a flat float32 shard, one elementwise pass: g = grad * grad_scale + weight_decay * p;
 * v = alpha v + (1 - alpha) g^2; p -= lr g / (sqrt(v) + eps).  With N ranks the step is reduce-scatter(grad) ->
 * idl_rmsprop_step on 1/N of the parameters -> all-gather(parameters). */
int idl_rmsprop_step(float* d_param, const float* d_grad, float* d_square_avg, int64_t n, float lr, float alpha, float eps, float weight_decay,
                     float grad_scale, void* stream);

/* The data-parallel optimiser step as ONE kernel over NVLink peer memory (gradient all-reduce + RMSprop + parameter
 * broadcast): gradients and parameters live in symmetric buffers, h_grad_peers / h_param_peers are HOST arrays of the `world`
 * device addresses at which this process sees every rank's buffer (entry `rank` = its own), grad_multicast / param_multicast the
 * NVLS multicast addresses of the same buffers or 0.  This rank reduces the slice [rank * n_total / world, +n_total / world) of
 * the gradients (multimem.ld_reduce when a multicast address is given: the switch adds the operands; otherwise one load per peer,
 * rank order), averages, applies idl_rmsprop_step's update to its slice (d_square_avg: n_total / world floats, local) and writes
 * the new parameters into every rank's buffer (multimem.st / one store per peer).  n_total % (4 * world) == 0, world <= 16.
 * The caller synchronises the ranks before (all gradients written) and after (all parameters visible) the call — two
 * symmetric-memory barriers of 5 us each; handshakes inside the kernel were measured slower (profiles/symm_probe_r2.txt). */
int idl_rmsprop_allreduce_step(const uint64_t* h_grad_peers, const uint64_t* h_param_peers, uint64_t grad_multicast, uint64_t param_multicast,
                               float* d_square_avg, int64_t n_total, int rank, int world, float lr, float alpha, float eps, float weight_decay,
                               void* stream);

/* The other two optimisers of idelucs/models.py:86-99 on a flat float32 shard, one elementwise pass each.  d_step points to the
 * 1-based number of the step being taken (int64 in device memory, 8-byte aligned): it is read by the kernel, so a replayed CUDA
 * graph keeps counting with the counter incremented on the device before the call.  g = grad * grad_scale + weight_decay * p.
 *   idl_sgd_step   torch.optim.SGD(lr, momentum, weight_decay), dampening 0, no Nesterov: buf = g at step 1, else
 *                  buf = momentum buf + g; p -= lr buf  (d_momentum_buf: n floats)
 *   idl_adam_step  torch.optim.Adam(lr, (beta1, beta2), eps, weight_decay), no amsgrad: m = m + (1 - beta1)(g - m);
 *                  v = beta2 v + (1 - beta2) g^2; p -= lr / (1 - beta1^t) m / (sqrt(v) / sqrt(1 - beta2^t) + eps), the bias
 *                  corrections in double; the betas are doubles, as torch holds them (1 - beta2 rounded from a float 0.999 is
 *                  1.3e-5 off)  (d_exp_avg, d_exp_avg_sq: n floats each) */
int idl_sgd_step(float* d_param, const float* d_grad, float* d_momentum_buf, int64_t n, float lr, float momentum, float weight_decay,
                 const int64_t* d_step, float grad_scale, void* stream);
int idl_adam_step(float* d_param, const float* d_grad, float* d_exp_avg, float* d_exp_avg_sq, int64_t n, float lr, double beta1, double beta2,
                  float eps, float weight_decay, const int64_t* d_step, float grad_scale, void* stream);

/* idl_rmsprop_allreduce_step with the SGD / Adam update: the same NVLink reduction and broadcast, the same argument rules (the
 * state buffers hold n_total / world floats each and are 16-byte aligned), the gradient mean taking the place of grad * grad_scale. */
int idl_sgd_allreduce_step(const uint64_t* h_grad_peers, const uint64_t* h_param_peers, uint64_t grad_multicast, uint64_t param_multicast,
                           float* d_momentum_buf, int64_t n_total, int rank, int world, float lr, float momentum, float weight_decay,
                           const int64_t* d_step, void* stream);
int idl_adam_allreduce_step(const uint64_t* h_grad_peers, const uint64_t* h_param_peers, uint64_t grad_multicast, uint64_t param_multicast,
                            float* d_exp_avg, float* d_exp_avg_sq, int64_t n_total, int rank, int world, float lr, double beta1, double beta2, float eps,
                            float weight_decay, const int64_t* d_step, void* stream);

/* F1 — FASTA ingest on the host (SURVEY §8f rank 1).  Replaces the record loop of kmersFasta
 * (idelucs/utils.py:229-261), which the reference re-runs on every pass (n_mimics + 1 times per training run,
 * once more per predict): '#' lines skipped (:230); a '>' line closes the running record only while its id is
 * non-empty (:233-252), then id = line[1:-1] (:253); other lines contribute line.strip() (:257); the last record
 * is always closed (:259-261).  Two calls over the file image `buf` (HOST memory):
 * idl_fasta_scan counts the records and the sequence bytes; idl_fasta_extract writes the concatenated sequence
 * bytes (seq_out, ideally pinned: it is what idl_pack reads after one H2D copy), byte_off int64[n_records+1],
 * and the id span of every record inside buf (hdr_off / hdr_len int64[n_records]).  The image is cut at line
 * boundaries and walked by up to 32 host threads; an idl_fasta_extract that directly follows idl_fasta_scan on the same
 * thread and image (which must not change in between) reuses its line index.  Alphabet handling
 * (check_sequence, :26-51) stays in idl_pack. */
int idl_fasta_scan(const uint8_t* buf, int64_t nbytes, int64_t* n_records, int64_t* n_seq_bytes);
int idl_fasta_extract(const uint8_t* buf, int64_t nbytes, int64_t n_records, uint8_t* seq_out, int64_t seq_cap,
                      int64_t* byte_off, int64_t* hdr_off, int64_t* hdr_len);

/* F3 — the all-pairs part of HDBSCAN (sklearn.cluster.HDBSCAN, Euclidean metric, alpha = 1), which the reference runs on
 * the latent vectors for --n_clusters 0 (idelucs/__main__.py:149-156).  d_x: float32 [n, D] row-major.  Distances are
 * computed exactly as sklearn does: the inputs widened to double, sum of (x_i[t] - x_j[t])^2 in order t = 0..D-1 with
 * every operation rounded on its own (no FMA), IEEE sqrt; results compare with sklearn's by ==.  d_ws:
 * idl_hdbscan_workspace_bytes(n, D) bytes (0 for n outside 1..2^31-1 or D < 1), 16-byte aligned, shared by both calls.
 * Memory is O(n D): no n x n matrix is stored, every pass recomputes the distances.
 * idl_core_distances: d_core[i] = the k-th smallest of the n distances d(i, .), counting d(i, i) = 0 and duplicates with
 *   multiplicity (NearestNeighbors.kneighbors(X, k)[0][:, -1]; sklearn's min_samples is k), 1 <= k <= n.  A radix select
 *   over the bit patterns of the squared distances: at most 9 launches, no host synchronisation.
 * idl_mreach_mst: the minimum spanning tree of the complete graph w(i, j) = max(d_core[i], d_core[j], d(i, j)) (sklearn's
 *   mst_from_data_matrix), with ties broken by (w, min(i, j), max(i, j)), so the tree is unique.  d_src, d_dst int64[n-1] and
 *   d_w double[n-1] receive its edges in the order Borůvka finds them (not sorted by weight), each oriented away from point 0
 *   (d_src is the endpoint on the path to point 0) as sklearn's Prim, grown from point 0, emits them.  The call
 *   SYNCHRONISES `stream` once per Borůvka round (at most ceil(log2 n) rounds: the components are merged on the host) and
 *   before it returns. */
size_t idl_hdbscan_workspace_bytes(int64_t n, int D);
int idl_core_distances(const float* d_x, int64_t n, int D, int64_t k, double* d_core, void* d_ws, size_t ws_bytes, void* stream);
int idl_mreach_mst(const float* d_x, const double* d_core, int64_t n, int D, int64_t* d_src, int64_t* d_dst, double* d_w, void* d_ws,
                   size_t ws_bytes, void* stream);
/* The same work split by rows, for one process driving several devices; results are bit-identical to the calls above.
 * idl_core_distances_rows: d_core[i] for the rows i of [row_begin, row_end) only (0 <= row_begin <= row_end <= n) of the
 *   full-length d_core; every row still takes its k-th smallest distance over all n columns.  Same workspace as above.
 * idl_mreach_mst_parts: idl_mreach_mst with every Borůvka round's all-pairs pass split into n_parts >= 1 row ranges
 *   [row_begin[p], row_end[p]) that partition [0, n) in order (empty parts allowed).  Part p runs on device devices[p] (a
 *   device may appear in several parts) with its own replicas d_x[p] and d_core[p] of the full x and core, its own workspace
 *   d_ws[p] (ws_bytes[p] >= idl_hdbscan_workspace_bytes(n, D)) and streams[p], a stream of that device.  Per round the host
 *   takes every component's lightest edge over the parts.  d_src / d_dst / d_w are written on devices[0] through
 *   streams[0].  All arrays are HOST arrays of n_parts entries.  The call SYNCHRONISES every part's stream once per round
 *   and streams[0] before it returns; the caller's current device is restored.  idl_mreach_mst is the one-part call on the
 *   current device. */
int idl_core_distances_rows(const float* d_x, int64_t n, int D, int64_t k, int64_t row_begin, int64_t row_end, double* d_core, void* d_ws,
                            size_t ws_bytes, void* stream);
int idl_mreach_mst_parts(int n_parts, const int* devices, const float* const* d_x, const double* const* d_core, const int64_t* row_begin,
                         const int64_t* row_end, int64_t n, int D, int64_t* d_src, int64_t* d_dst, double* d_w, void* const* d_ws,
                         const size_t* ws_bytes, void* const* streams);

/* F4 — per-sample silhouette coefficients (sklearn.metrics.silhouette_samples, Euclidean metric), the internal
 * clustering metric the reference writes to metrics.tsv (idelucs/utils.py compute_results).  d_x: float32 [n, D]
 * row-major; d_labels: int32 [n], every label in 0..n_labels-1 (empty labels are allowed); d_out: double [n].
 * Arithmetic (results compare with a sequential fp64 reference by ==):
 *   d(i, j)  = exactly the distance of idl_core_distances: inputs widened to double, sum of (x_i[t] - x_j[t])^2 in order
 *              t = 0..D-1 with every operation rounded on its own (no FMA), IEEE sqrt;
 *   S_c(i)   = ((0 + d(i, j1)) + d(i, j2)) + ... over the points j1 < j2 < ... of cluster c, self included (d(i, i) = 0);
 *   intra    = S_own / (n_own - 1);  inter = min over non-empty c != own of S_c / n_c;
 *   s(i)     = (inter - intra) / max(intra, inter), and 0 when n_own = 1 or the quotient is NaN (intra = inter = 0, or no
 *              other non-empty cluster): sklearn's nan_to_num.
 * d_ws: idl_silhouette_workspace_bytes(n, n_labels) bytes (0 for n outside 1..2^31-1 or n_labels outside 1..n),
 * 16-byte aligned; memory is O(n D + n): no n x n matrix is stored.  The call copies the labels to the host and
 * SYNCHRONISES `stream` once, before any kernel runs: a label outside 0..n_labels-1 returns IDL_EINVAL naming its
 * position.  The host groups the points by label (stable counting sort) and one all-pairs kernel follows, enqueued
 * on `stream` (d_out is ready when `stream` is). */
size_t idl_silhouette_workspace_bytes(int64_t n, int64_t n_labels);
int idl_silhouette_samples(const float* d_x, const int32_t* d_labels, int64_t n, int D, int64_t n_labels, double* d_out, void* d_ws,
                           size_t ws_bytes, void* stream);
/* the same for the rows of [row_begin, row_end) only (0 <= row_begin <= row_end <= n): d_out[i] for those rows of the
 * full-length d_out, each row still against all n columns; the grouping, the label check and the synchronisation are those of
 * idl_silhouette_samples.  Split over devices, every call computes bits identical to the one-call result. */
int idl_silhouette_samples_rows(const float* d_x, const int32_t* d_labels, int64_t n, int D, int64_t n_labels, int64_t row_begin,
                                int64_t row_end, double* d_out, void* d_ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IDELUCS_B200_H */
