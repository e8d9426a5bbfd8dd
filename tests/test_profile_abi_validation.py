"""Argument validation of the k-mer profile entry points of the C ABI (idl_profiles, idl_profiles_chunked,
idl_profiles_prepared, idl_profiles_prepare, idl_profile_stats, idl_kmer_counts and the two sizing functions): the
return code and the exact idl_last_error() text of every argument set in the tables below.

The calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that passes validation fails at its first
CUDA call with IDL_ECUDA instead of launching on the placeholder pointers: the tables also pin where validation ends.
Placeholder device pointers are small aligned integers; the host code never dereferences them."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, 1, 2, 3
CLEAN, TRANSITION, TRANSVERSION, BOTH, RANDOM_N, EXPLICIT = range(6)
COUNTS_I32, FREQ_F32, STD_F32, FREQ_F64 = range(4)
DEV = 64   # placeholder device pointer (16-byte aligned)

# (kind, p1, p2, n_bp) per variant
SCHEDULE = [(BOTH, 1e-2, 5e-3, 0), (TRANSITION, 1e-2, 0.0, 0), (TRANSVERSION, 0.0, 5e-3, 0), (RANDOM_N, 0.0, 0.0, 20)]

# argument order of each entry point (include/idelucs_b200.h)
ORDER = {
    "idl_profiles": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants sel S seed edit_off edits out_kind "
                    "out out_off out_stride pseudocount accumulate mean scale status ws ws_bytes stream",
    "idl_profiles_chunked": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants sel S seed edit_off edits "
                            "out_kind out out_off out_stride pseudocount accumulate mean scale scratch scratch_bytes max_long ws "
                            "ws_bytes stream",
    "idl_profiles_prepared": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants seed out_kind out out_off "
                             "out_stride pseudocount mean scale status prep prep_size ws ws_bytes stream",
    "idl_profiles_prepare": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants seed pseudocount prep "
                            "prep_size partials part_n max_parts n_parts status ws ws_bytes stream",
    "idl_profile_stats": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants seed edit_off edits pseudocount partials "
                         "part_n max_parts n_parts status ws ws_bytes stream",
    "idl_kmer_counts": "codes nmask chunk_off len n_items k out accumulate ws ws_bytes stream",
    "idl_profiles_chunked_bytes": "n_items max_long variants n_variants S",
    "idl_prepare_bytes": "n_items",
}
BASE = dict(codes=DEV, nmask=DEV, chunk_off=DEV, len=DEV, n_seqs=1000, sidx=None, n_items=1000, seq_id0=0, k=6, variants=SCHEDULE,
            sel=None, seed=12345, edit_off=None, edits=None, out_kind=FREQ_F32, out=DEV, out_stride=4096, pseudocount=1, accumulate=0,
            mean=None, scale=None, status=None, ws=DEV, ws_bytes="ws", stream=None, scratch=DEV, scratch_bytes=1 << 30, max_long=2,
            prep=DEV, prep_size="prep", partials=DEV, part_n=DEV, max_parts=2048, n_parts=-1)
PER_ENTRY = {
    "idl_profiles_prepared": dict(status=DEV),
    "idl_profiles_prepare": dict(status=DEV),
    "idl_profile_stats": dict(variants=[(CLEAN, 0.0, 0.0, 0)]),
    "idl_kmer_counts": dict(out_kind=COUNTS_I32),
}
POINTERS = set("codes nmask chunk_off len sidx sel edit_off edits out mean scale status ws stream scratch prep partials part_n".split())

NULL = "idl_profiles: null pointer"
WS_SMALL = "idl_profiles: workspace too small (need {ws} bytes)"
CUDA = "<cuda>"   # any CUDA runtime error: the request got past validation
ALIGN = "idl_profiles: d_out must be 16-byte aligned and out_off multiples of 4"

# (id, entry point, arguments that differ from BASE / PER_ENTRY, (return code, error text or CUDA or None))
CASES = [
    ("valid", "idl_profiles", {}, (ECUDA, CUDA)),
    ("valid_counts_accumulate", "idl_profiles", dict(out_kind=COUNTS_I32, accumulate=1), (ECUDA, CUDA)),
    ("valid_cta_cap_bits", "idl_profiles", dict(accumulate=3 << 8), (ECUDA, CUDA)),
    ("valid_std", "idl_profiles", dict(out_kind=STD_F32, mean=DEV, scale=DEV), (ECUDA, CUDA)),
    ("valid_f64", "idl_profiles", dict(out_kind=FREQ_F64), (ECUDA, CUDA)),
    ("valid_sel", "idl_profiles", dict(sel=DEV, S=2), (ECUDA, CUDA)),
    ("valid_k1", "idl_profiles", dict(k=1, out_stride=4), (ECUDA, CUDA)),
    ("valid_explicit_with_lists", "idl_profiles", dict(variants=[(EXPLICIT, 0.0, 0.0, 0)], edit_off=DEV, edits=DEV), (ECUDA, CUDA)),
    ("valid_random_n_1024", "idl_profiles", dict(variants=[(RANDOM_N, 0.0, 0.0, 1024)]), (ECUDA, CUDA)),
    ("valid_big_plan_65_variants", "idl_profiles", dict(variants=[(CLEAN, 0.0, 0.0, 0)] * 65), (ECUDA, CUDA)),
    ("valid_64_rates", "idl_profiles", dict(variants=[(BOTH, 0.001 * i, 0.5 + 0.001 * i, 0) for i in range(32)]), (ECUDA, CUDA)),
    ("null_codes", "idl_profiles", dict(codes=None), (EINVAL, NULL)),
    ("null_nmask", "idl_profiles", dict(nmask=None), (EINVAL, NULL)),
    ("null_chunk_off", "idl_profiles", dict(chunk_off=None), (EINVAL, NULL)),
    ("null_len", "idl_profiles", dict(len=None), (EINVAL, NULL)),
    ("null_variants", "idl_profiles", dict(variants=None, n_variants=4), (EINVAL, NULL)),
    ("null_out", "idl_profiles", dict(out=None), (EINVAL, NULL)),
    ("null_out_off", "idl_profiles", dict(out_off=None), (EINVAL, NULL)),
    ("null_workspace", "idl_profiles", dict(ws=None), (EINVAL, NULL)),
    ("workspace_too_small", "idl_profiles", dict(ws_bytes="ws-1"), (EINVAL, WS_SMALL)),
    ("k0", "idl_profiles", dict(k=0), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 0)")),
    ("k7", "idl_profiles", dict(k=7), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),
    ("n_variants_0", "idl_profiles", dict(n_variants=0, S=4), (EINVAL, "idl_profiles: n_variants / S out of range")),
    ("n_variants_4097", "idl_profiles", dict(variants=[(CLEAN, 0.0, 0.0, 0)] * 4097), (EINVAL, "idl_profiles: n_variants / S out of range")),
    ("S_0", "idl_profiles", dict(sel=DEV, S=0, out_off=[0]), (EINVAL, "idl_profiles: n_variants / S out of range")),
    ("S_4097", "idl_profiles", dict(sel=DEV, S=4097), (EINVAL, "idl_profiles: n_variants / S out of range")),
    ("S_without_sel", "idl_profiles", dict(S=3), (EINVAL, "idl_profiles: S must equal n_variants without d_sel")),
    ("std_without_mean", "idl_profiles", dict(out_kind=STD_F32, scale=DEV), (EINVAL, "idl_profiles: mean/scale required")),
    ("std_without_scale", "idl_profiles", dict(out_kind=STD_F32, mean=DEV), (EINVAL, "idl_profiles: mean/scale required")),
    ("accumulate_freq", "idl_profiles", dict(accumulate=1), (EINVAL, "idl_profiles: accumulate only for counts")),
    ("accumulate_f64", "idl_profiles", dict(out_kind=FREQ_F64, accumulate=1 | (2 << 8)), (EINVAL, "idl_profiles: accumulate only for counts")),
    ("out_kind_4", "idl_profiles", dict(out_kind=4), (EINVAL, "idl_profiles: unknown out_kind 4")),
    ("out_kind_negative", "idl_profiles", dict(out_kind=-1, out=None), (EINVAL, "idl_profiles: unknown out_kind -1")),
    ("n_items_0", "idl_profiles", dict(n_items=0), (OK, None)),
    ("n_items_negative", "idl_profiles", dict(n_items=-5, out_stride=3), (OK, None)),
    ("n_items_0_still_checks_k", "idl_profiles", dict(n_items=0, k=7), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),
    ("out_stride_not_multiple_of_4", "idl_profiles", dict(out_stride=4098), (EINVAL, "idl_profiles: out_stride must be a multiple of 4")),
    ("out_misaligned", "idl_profiles", dict(out=68), (EINVAL, ALIGN)),
    ("out_8_aligned_f64", "idl_profiles", dict(out=72, out_kind=FREQ_F64), (EINVAL, ALIGN)),
    ("out_off_not_multiple_of_4", "idl_profiles", dict(out_off=[0, 0, 2, 0]), (EINVAL, ALIGN)),
    ("out_off_multiple_of_4", "idl_profiles", dict(out_off=[4, 8, 12, 4096]), (ECUDA, CUDA)),
    ("bad_kind_6", "idl_profiles", dict(variants=[(CLEAN, 0.0, 0.0, 0), (6, 0.0, 0.0, 0)]), (EINVAL, "idl_profiles: bad variant kind 6")),
    ("bad_kind_negative", "idl_profiles", dict(variants=[(-1, 0.0, 0.0, 0)]), (EINVAL, "idl_profiles: bad variant kind -1")),
    ("p1_above_1", "idl_profiles", dict(variants=[(TRANSITION, 1.5, 0.0, 0)]), (EINVAL, "idl_profiles: p1 out of range")),
    ("p1_nan", "idl_profiles", dict(variants=[(BOTH, float("nan"), 0.1, 0)]), (EINVAL, "idl_profiles: p1 out of range")),
    ("p2_negative", "idl_profiles", dict(variants=[(TRANSVERSION, 0.0, -0.1, 0)]), (EINVAL, "idl_profiles: p2 out of range")),
    ("p2_of_both", "idl_profiles", dict(variants=[(BOTH, 0.1, 2.0, 0)]), (EINVAL, "idl_profiles: p2 out of range")),
    ("p1_ignored_for_transversion", "idl_profiles", dict(variants=[(TRANSVERSION, 7.0, 0.1, 0)]), (ECUDA, CUDA)),
    ("too_many_rates", "idl_profiles", dict(variants=[(BOTH, 0.001 * i, 0.5 + 0.001 * i, 0) for i in range(33)]),
     (EUNSUPPORTED, "idl_profiles: too many distinct mutation rates")),
    ("random_n_1025", "idl_profiles", dict(variants=[(RANDOM_N, 0.0, 0.0, 1025)]), (EUNSUPPORTED, "idl_profiles: Random_N n_bp must be <= 1024")),
    ("random_n_negative", "idl_profiles", dict(variants=[(RANDOM_N, 0.0, 0.0, -1)]), (EUNSUPPORTED, "idl_profiles: Random_N n_bp must be <= 1024")),
    ("explicit_without_lists", "idl_profiles", dict(variants=[(EXPLICIT, 0.0, 0.0, 0)], edit_off=DEV),
     (EINVAL, "idl_profiles: explicit variant without edit lists")),

    ("valid", "idl_profiles_chunked", {}, (ECUDA, CUDA)),
    ("valid_max_long_0", "idl_profiles_chunked", dict(max_long=0, out_kind=COUNTS_I32, accumulate=1), (ECUDA, CUDA)),
    ("out_kind_4", "idl_profiles_chunked", dict(out_kind=4), (EINVAL, "idl_profiles_chunked: unknown out_kind 4")),
    ("no_scratch", "idl_profiles_chunked", dict(scratch=None), (EINVAL, "idl_profiles_chunked: scratch required")),
    ("max_long_negative", "idl_profiles_chunked", dict(max_long=-1), (EINVAL, "idl_profiles_chunked: scratch required")),
    ("null_codes", "idl_profiles_chunked", dict(codes=None), (EINVAL, NULL)),
    ("workspace_too_small", "idl_profiles_chunked", dict(ws_bytes="ws-1"), (EINVAL, WS_SMALL)),
    ("k7", "idl_profiles_chunked", dict(k=7), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),
    ("S_without_sel", "idl_profiles_chunked", dict(S=5), (EINVAL, "idl_profiles: S must equal n_variants without d_sel")),
    ("std_without_mean", "idl_profiles_chunked", dict(out_kind=STD_F32), (EINVAL, "idl_profiles: mean/scale required")),
    ("accumulate_freq", "idl_profiles_chunked", dict(accumulate=1), (EINVAL, "idl_profiles: accumulate only for counts")),
    ("bad_kind", "idl_profiles_chunked", dict(variants=[(9, 0.0, 0.0, 0)]), (EINVAL, "idl_profiles: bad variant kind 9")),
    ("n_items_0", "idl_profiles_chunked", dict(n_items=0), (OK, None)),
    ("out_misaligned", "idl_profiles_chunked", dict(out=84, out_kind=COUNTS_I32), (EINVAL, ALIGN)),

    ("valid", "idl_profiles_prepared", {}, (ECUDA, CUDA)),
    ("valid_std", "idl_profiles_prepared", dict(out_kind=STD_F32, mean=DEV, scale=DEV), (ECUDA, CUDA)),
    ("counts", "idl_profiles_prepared", dict(out_kind=COUNTS_I32), (EINVAL, "idl_profiles_prepared: float32 outputs only")),
    ("f64", "idl_profiles_prepared", dict(out_kind=FREQ_F64), (EINVAL, "idl_profiles_prepared: float32 outputs only")),
    ("no_prep", "idl_profiles_prepared", dict(prep=None), (EINVAL, "idl_profiles_prepared: d_prep and d_status are required")),
    ("no_status", "idl_profiles_prepared", dict(status=None), (EINVAL, "idl_profiles_prepared: d_prep and d_status are required")),
    ("null_out", "idl_profiles_prepared", dict(out=None), (EINVAL, NULL)),
    ("workspace_too_small", "idl_profiles_prepared", dict(ws_bytes="ws-1"), (EINVAL, WS_SMALL)),
    ("k0", "idl_profiles_prepared", dict(k=0), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 0)")),
    ("std_without_scale", "idl_profiles_prepared", dict(out_kind=STD_F32, mean=DEV), (EINVAL, "idl_profiles: mean/scale required")),
    ("explicit", "idl_profiles_prepared", dict(variants=[(EXPLICIT, 0.0, 0.0, 0)]), (EINVAL, "idl_profiles: explicit variant without edit lists")),
    ("n_items_0", "idl_profiles_prepared", dict(n_items=0), (OK, None)),
    ("out_misaligned", "idl_profiles_prepared", dict(out=68), (EINVAL, ALIGN)),
    ("out_off_not_multiple_of_4", "idl_profiles_prepared", dict(out_off=[0, 0, 0, 4098]), (EINVAL, ALIGN)),

    ("valid", "idl_profiles_prepare", {}, (ECUDA, CUDA)),
    ("valid_without_statistics", "idl_profiles_prepare", dict(partials=None, part_n=None, max_parts=0, n_parts=None), (ECUDA, CUDA)),
    ("valid_random_n_slot0_without_draws", "idl_profiles_prepare", dict(variants=[(RANDOM_N, 0.0, 0.0, 0)] + SCHEDULE), (ECUDA, CUDA)),
    ("valid_64_variants", "idl_profiles_prepare", dict(variants=SCHEDULE + [(RANDOM_N, 0.0, 0.0, 20)] * 60), (ECUDA, CUDA)),
    ("valid_max_parts_1184", "idl_profiles_prepare", dict(max_parts=1184), (ECUDA, CUDA)),
    ("five_rates_plan_copied_first", "idl_profiles_prepare", dict(variants=[(BOTH, 0.1, 0.2, 0), (BOTH, 0.3, 0.4, 0), (TRANSITION, 0.5, 0.0, 0)]),
     (ECUDA, CUDA)),
    ("null_codes", "idl_profiles_prepare", dict(codes=None), (EINVAL, "idl_profiles_prepare: null pointer")),
    ("null_variants", "idl_profiles_prepare", dict(variants=None, n_variants=4), (EINVAL, "idl_profiles_prepare: null pointer")),
    ("null_prep", "idl_profiles_prepare", dict(prep=None), (EINVAL, "idl_profiles_prepare: null pointer")),
    ("null_status", "idl_profiles_prepare", dict(status=None), (EINVAL, "idl_profiles_prepare: null pointer")),
    ("null_workspace", "idl_profiles_prepare", dict(ws=None), (EINVAL, "idl_profiles_prepare: null pointer")),
    ("k5", "idl_profiles_prepare", dict(k=5), (EUNSUPPORTED, "idl_profiles_prepare: k must be 6 (got 5)")),
    ("workspace_too_small", "idl_profiles_prepare", dict(ws_bytes="ws-1"), (EINVAL, "idl_profiles_prepare: workspace too small (need {ws} bytes)")),
    ("n_variants_0", "idl_profiles_prepare", dict(n_variants=0), (EUNSUPPORTED, "idl_profiles_prepare: 1..64 variants")),
    ("n_variants_65", "idl_profiles_prepare", dict(variants=SCHEDULE + [(RANDOM_N, 0.0, 0.0, 20)] * 61), (EUNSUPPORTED, "idl_profiles_prepare: 1..64 variants")),
    ("n_items_0", "idl_profiles_prepare", dict(n_items=0, prep_size=0, max_parts=0), (OK, None)),
    ("n_items_0_no_n_parts", "idl_profiles_prepare", dict(n_items=0, n_parts=None), (OK, None)),
    ("n_items_0_still_checks_k", "idl_profiles_prepare", dict(n_items=0, k=4), (EUNSUPPORTED, "idl_profiles_prepare: k must be 6 (got 4)")),
    ("prep_too_small", "idl_profiles_prepare", dict(prep_size="prep-1"), (EINVAL, "idl_profiles_prepare: d_prep too small (need {prep} bytes)")),
    ("prep_misaligned", "idl_profiles_prepare", dict(prep=72), (EINVAL, "idl_profiles_prepare: misaligned buffer")),
    ("codes_misaligned", "idl_profiles_prepare", dict(codes=72), (EINVAL, "idl_profiles_prepare: misaligned buffer")),
    ("nmask_misaligned", "idl_profiles_prepare", dict(nmask=68), (EINVAL, "idl_profiles_prepare: misaligned buffer")),
    ("nmask_8_aligned", "idl_profiles_prepare", dict(nmask=72), (ECUDA, CUDA)),
    ("statistics_without_part_n", "idl_profiles_prepare", dict(part_n=None),
     (EINVAL, "idl_profiles_prepare: statistics need d_part_n, n_parts and max_parts >= 8 x SMs")),
    ("statistics_without_n_parts", "idl_profiles_prepare", dict(n_parts=None),
     (EINVAL, "idl_profiles_prepare: statistics need d_part_n, n_parts and max_parts >= 8 x SMs")),
    ("statistics_max_parts_1183", "idl_profiles_prepare", dict(max_parts=1183),
     (EINVAL, "idl_profiles_prepare: statistics need d_part_n, n_parts and max_parts >= 8 x SMs")),
    ("bad_kind", "idl_profiles_prepare", dict(variants=[(CLEAN, 0.0, 0.0, 0), (8, 0.0, 0.0, 0)]), (EINVAL, "idl_profiles_prepare: bad variant kind 8")),
    ("p1_out_of_range", "idl_profiles_prepare", dict(variants=[(TRANSITION, -1.0, 0.0, 0)]), (EINVAL, "idl_profiles_prepare: p1 out of range")),
    ("p2_out_of_range", "idl_profiles_prepare", dict(variants=[(BOTH, 0.1, 1.5, 0)]), (EINVAL, "idl_profiles_prepare: p2 out of range")),
    ("too_many_rates", "idl_profiles_prepare", dict(variants=[(BOTH, 0.001 * i, 0.5 + 0.001 * i, 0) for i in range(33)]),
     (EUNSUPPORTED, "idl_profiles_prepare: too many distinct mutation rates")),
    ("random_n_1025", "idl_profiles_prepare", dict(variants=[(CLEAN, 0.0, 0.0, 0), (RANDOM_N, 0.0, 0.0, 1025)]),
     (EUNSUPPORTED, "idl_profiles_prepare: Random_N n_bp must be <= 1024")),
    ("explicit", "idl_profiles_prepare", dict(variants=[(CLEAN, 0.0, 0.0, 0), (EXPLICIT, 0.0, 0.0, 0)]),
     (EINVAL, "idl_profiles_prepare: explicit variant without edit lists")),
    ("four_bernoulli_slots", "idl_profiles_prepare", dict(variants=SCHEDULE + [(TRANSITION, 1e-2, 0.0, 0)]),
     (EUNSUPPORTED, "idl_profiles_prepare: at most 3 Bernoulli slots, 4 distinct rates, no explicit lists")),
    ("random_n_slot0", "idl_profiles_prepare", dict(variants=[(RANDOM_N, 0.0, 0.0, 20)] + SCHEDULE[:3]),
     (EUNSUPPORTED, "idl_profiles_prepare: slot 0 must be clean or a Bernoulli mimic")),

    ("valid", "idl_profile_stats", {}, (ECUDA, CUDA)),
    ("valid_bernoulli", "idl_profile_stats", dict(variants=[(BOTH, 1e-2, 5e-3, 0)], k=4), (ECUDA, CUDA)),
    ("valid_explicit_with_lists", "idl_profile_stats", dict(variants=[(EXPLICIT, 0.0, 0.0, 0)], edit_off=DEV, edits=DEV), (ECUDA, CUDA)),
    ("valid_max_parts_1184", "idl_profile_stats", dict(max_parts=1184), (ECUDA, CUDA)),
    ("null_partials", "idl_profile_stats", dict(partials=None), (EINVAL, "idl_profile_stats: null pointer")),
    ("null_part_n", "idl_profile_stats", dict(part_n=None), (EINVAL, "idl_profile_stats: null pointer")),
    ("null_n_parts", "idl_profile_stats", dict(n_parts=None), (EINVAL, "idl_profile_stats: null pointer")),
    ("null_variant", "idl_profile_stats", dict(variants=None), (EINVAL, "idl_profile_stats: null pointer")),
    ("max_parts_1183", "idl_profile_stats", dict(max_parts=1183), (EINVAL, "idl_profile_stats: max_parts too small (need 1184)")),
    ("n_items_0", "idl_profile_stats", dict(n_items=0), (OK, None)),
    ("n_items_0_still_checks_max_parts", "idl_profile_stats", dict(n_items=0, max_parts=8), (EINVAL, "idl_profile_stats: max_parts too small (need 1184)")),
    ("null_codes", "idl_profile_stats", dict(codes=None), (EINVAL, NULL)),
    ("workspace_too_small", "idl_profile_stats", dict(ws_bytes="ws-1"), (EINVAL, WS_SMALL)),
    ("k7", "idl_profile_stats", dict(k=7), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),
    ("bad_kind", "idl_profile_stats", dict(variants=[(7, 0.0, 0.0, 0)]), (EINVAL, "idl_profiles: bad variant kind 7")),
    ("p1_out_of_range", "idl_profile_stats", dict(variants=[(TRANSITION, 2.0, 0.0, 0)]), (EINVAL, "idl_profiles: p1 out of range")),
    ("random_n_1025", "idl_profile_stats", dict(variants=[(RANDOM_N, 0.0, 0.0, 1025)]), (EUNSUPPORTED, "idl_profiles: Random_N n_bp must be <= 1024")),
    ("explicit_without_lists", "idl_profile_stats", dict(variants=[(EXPLICIT, 0.0, 0.0, 0)], edits=DEV),
     (EINVAL, "idl_profiles: explicit variant without edit lists")),

    ("valid", "idl_kmer_counts", {}, (ECUDA, CUDA)),
    ("valid_accumulate", "idl_kmer_counts", dict(accumulate=1, k=3), (ECUDA, CUDA)),
    ("k0", "idl_kmer_counts", dict(k=0), (EUNSUPPORTED, "idl_kmer_counts: k must be in 1..6 (got 0)")),
    ("k7", "idl_kmer_counts", dict(k=7), (EUNSUPPORTED, "idl_kmer_counts: k must be in 1..6 (got 7)")),
    ("null_codes", "idl_kmer_counts", dict(codes=None), (EINVAL, NULL)),
    ("null_counts", "idl_kmer_counts", dict(out=None), (EINVAL, NULL)),
    ("null_workspace", "idl_kmer_counts", dict(ws=None), (EINVAL, NULL)),
    ("workspace_too_small", "idl_kmer_counts", dict(ws_bytes="ws-1"), (EINVAL, WS_SMALL)),
    ("n_0", "idl_kmer_counts", dict(n_items=0), (OK, None)),
]

# the sizing functions: (id, entry point, arguments, expected result); without a device the chunked path has no grid to size
SIZES = [
    ("valid_without_device", "idl_profiles_chunked_bytes", {}, 0),
    ("seven_dense", "idl_profiles_chunked_bytes", dict(variants=[(BOTH, 0.1, 0.1, 0)] * 8, S=7), 0),
    ("eight_dense", "idl_profiles_chunked_bytes", dict(variants=[(BOTH, 0.1, 0.1, 0)] * 8), 0),
    ("n_items_0", "idl_profiles_chunked_bytes", dict(n_items=0), 0),
    ("max_long_0", "idl_profiles_chunked_bytes", dict(max_long=0), 0),
    ("null_variants", "idl_profiles_chunked_bytes", dict(variants=None, n_variants=4), 0),
    ("n_variants_0", "idl_profiles_chunked_bytes", dict(n_variants=0), 0),
    ("S_0", "idl_profiles_chunked_bytes", dict(S=0), 0),
    ("n_items_0", "idl_prepare_bytes", dict(n_items=0), 0),
    ("n_items_negative", "idl_prepare_bytes", dict(n_items=-3), 0),
]


def _call_all():
    """child process: run every case, return {case key: [rc, error text, n_parts]} and the sizes the texts quote"""
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    ws_total = lib.idl_profiles_workspace_bytes()

    def call(entry, over):
        a = dict(BASE, **PER_ENTRY.get(entry, {}))
        a.update(over)
        if a["variants"] is not None:
            a.setdefault("n_variants", len(a["variants"]))
        a.setdefault("n_variants", 1)
        a.setdefault("S", a["n_variants"])
        a.setdefault("out_off", [0] * max(a["S"], 1))
        a["ws_bytes"] = {"ws": ws_total, "ws-1": ws_total - 1}.get(a["ws_bytes"], a["ws_bytes"])
        prep = lib.idl_prepare_bytes(a["n_items"])
        a["prep_size"] = {"prep": prep, "prep-1": prep - 1}.get(a["prep_size"], a["prep_size"])
        n_parts = None if a["n_parts"] is None else ctypes.c_int(a["n_parts"])
        args = []
        for name in ORDER[entry].split():
            v = a[name]
            if name == "variants" and v is not None:
                arr = (_lib.Variant * len(v))()
                for i, (kind, p1, p2, n_bp) in enumerate(v):
                    arr[i].kind, arr[i].rng_id, arr[i].n_bp, arr[i].explicit_idx, arr[i].p1, arr[i].p2 = kind, i, n_bp, 0, p1, p2
                v = arr
            elif name == "out_off" and v is not None:
                v = (ctypes.c_int64 * len(v))(*v)
            elif name == "n_parts" and v is not None:
                v = ctypes.byref(n_parts)
            elif name in POINTERS and v is not None:
                v = ctypes.c_void_p(v)
            args.append(v)
        rc = getattr(lib, entry)(*args)
        return [rc, lib.idl_last_error().decode(), None if n_parts is None else n_parts.value], prep

    out, prep = {}, {}
    for cid, entry, over, _ in CASES:
        out[entry + "::" + cid], prep[entry + "::" + cid] = call(entry, over)
    for cid, entry, over, _ in SIZES:
        out[entry + "::" + cid] = [call(entry, over)[0][0]]
    sizes = [lib.idl_prepare_bytes(n) for n in (1, 2, 1000, 10 ** 6)]
    return {"ws": ws_total, "prep": prep, "results": out, "prepare_bytes": sizes}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("case", CASES, ids=[c[1] + "::" + c[0] for c in CASES])
def test_profile_entry_point_validation(called, case):
    cid, entry, over, (rc, text) = case
    key = entry + "::" + cid
    got_rc, got_text, n_parts = called["results"][key]
    assert got_rc == rc, (key, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    elif text is not None:
        assert got_text == text.format(ws=called["ws"], prep=called["prep"][key])
    if rc == OK and entry in ("idl_profiles_prepare", "idl_profile_stats") and over.get("n_parts", BASE["n_parts"]) is not None:
        assert n_parts == 0   # nothing to do: no parts written


@pytest.mark.parametrize("case", SIZES, ids=[c[1] + "::" + c[0] for c in SIZES])
def test_profile_sizing_functions(called, case):
    cid, entry, _, want = case
    assert called["results"][entry + "::" + cid] == [want]


def test_prepare_bytes_grow_with_the_items(called):
    sizes = called["prepare_bytes"]
    assert all(0 < a < b for a, b in zip(sizes, sizes[1:])), sizes


if __name__ == "__main__":
    print(json.dumps(_call_all()))
