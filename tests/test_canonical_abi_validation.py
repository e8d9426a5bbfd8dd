"""Argument validation of the canonical output kinds (IDL_OUT_CANON_F32 / _STD_F32 / _F64) at the profile entry points:
the return code and the exact idl_last_error() text of every argument set below.

Like test_profile_abi_validation.py, the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that
passes validation fails at its first CUDA call with IDL_ECUDA instead of launching on the placeholder pointers."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, 1, 2, 3
CLEAN, TRANSITION, TRANSVERSION, BOTH, RANDOM_N, EXPLICIT = range(6)
FREQ_F32, STD_F32 = 1, 2
CANON_F32, CANON_STD_F32, CANON_F64 = 9, 10, 11
DEV = 64   # placeholder device pointer (16-byte aligned)
SCHEDULE = [(BOTH, 1e-2, 5e-3, 0), (TRANSITION, 1e-2, 0.0, 0), (TRANSVERSION, 0.0, 5e-3, 0), (RANDOM_N, 0.0, 0.0, 20)]

ORDER = {
    "idl_profiles": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants sel S seed edit_off edits out_kind "
                    "out out_off out_stride pseudocount accumulate mean scale status ws ws_bytes stream",
    "idl_profiles_chunked": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants sel S seed edit_off edits "
                            "out_kind out out_off out_stride pseudocount accumulate mean scale scratch scratch_bytes max_long ws "
                            "ws_bytes stream",
    "idl_profiles_prepared": "codes nmask chunk_off len n_seqs sidx n_items seq_id0 k variants n_variants seed out_kind out out_off "
                             "out_stride pseudocount mean scale status prep prep_size ws ws_bytes stream",
}
BASE = dict(codes=DEV, nmask=DEV, chunk_off=DEV, len=DEV, n_seqs=1000, sidx=None, n_items=1000, seq_id0=0, k=6, variants=SCHEDULE,
            sel=None, seed=12345, edit_off=None, edits=None, out_kind=CANON_F32, out=DEV, out_stride=2080, pseudocount=1, accumulate=0,
            mean=None, scale=None, status=DEV, ws=DEV, ws_bytes="ws", stream=None, scratch=DEV, scratch_bytes=1 << 30, max_long=2,
            prep=DEV, prep_size="prep")
POINTERS = set("codes nmask chunk_off len sidx sel edit_off edits out mean scale status ws stream scratch prep".split())
CUDA = "<cuda>"   # any CUDA runtime error: the request got past validation
PREPARED = "idl_profiles_prepared: canonical output kinds are not supported (use idl_profiles or idl_profiles_chunked)"
MEAN = "idl_profiles: mean/scale required"

CASES = [
    ("valid_f32", "idl_profiles", {}, (ECUDA, CUDA)),
    ("valid_f64", "idl_profiles", dict(out_kind=CANON_F64), (ECUDA, CUDA)),
    ("valid_std", "idl_profiles", dict(out_kind=CANON_STD_F32, mean=DEV, scale=DEV), (ECUDA, CUDA)),
    ("valid_k1_odd_stride_and_offset", "idl_profiles", dict(k=1, out_stride=3, out_off=[5] * 4), (ECUDA, CUDA)),
    ("valid_k2_stride_10", "idl_profiles", dict(k=2, out_stride=10, out_kind=CANON_F64), (ECUDA, CUDA)),
    ("valid_sel", "idl_profiles", dict(sel=DEV, S=2, sidx=DEV), (ECUDA, CUDA)),
    ("std_without_mean", "idl_profiles", dict(out_kind=CANON_STD_F32, scale=DEV), (EINVAL, MEAN)),
    ("std_without_scale", "idl_profiles", dict(out_kind=CANON_STD_F32, mean=DEV), (EINVAL, MEAN)),
    ("std_without_either_n_items_0", "idl_profiles", dict(out_kind=CANON_STD_F32, n_items=0), (EINVAL, MEAN)),
    ("accumulate", "idl_profiles", dict(accumulate=1), (EINVAL, "idl_profiles: accumulate only for counts")),
    ("out_kind_8", "idl_profiles", dict(out_kind=8), (EINVAL, "idl_profiles: unknown out_kind 8")),
    ("out_kind_12", "idl_profiles", dict(out_kind=12), (EINVAL, "idl_profiles: unknown out_kind 12")),
    ("k0", "idl_profiles", dict(k=0), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 0)")),
    ("k7", "idl_profiles", dict(k=7), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),
    ("k7_std", "idl_profiles", dict(k=7, out_kind=CANON_STD_F32, mean=DEV, scale=DEV), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),

    ("valid_f32", "idl_profiles_chunked", {}, (ECUDA, CUDA)),
    ("valid_std_odd_stride", "idl_profiles_chunked", dict(out_kind=CANON_STD_F32, mean=DEV, scale=DEV, out_stride=2081), (ECUDA, CUDA)),
    ("std_without_mean", "idl_profiles_chunked", dict(out_kind=CANON_STD_F32, scale=DEV), (EINVAL, MEAN)),
    ("out_kind_12", "idl_profiles_chunked", dict(out_kind=12), (EINVAL, "idl_profiles_chunked: unknown out_kind 12")),
    ("k7", "idl_profiles_chunked", dict(k=7, out_kind=CANON_F64), (EUNSUPPORTED, "idl_profiles: k must be in 1..6 (got 7)")),

    ("canon_f32", "idl_profiles_prepared", {}, (EINVAL, PREPARED)),
    ("canon_std", "idl_profiles_prepared", dict(out_kind=CANON_STD_F32, mean=DEV, scale=DEV), (EINVAL, PREPARED)),
    ("canon_f64", "idl_profiles_prepared", dict(out_kind=CANON_F64), (EINVAL, PREPARED)),
    ("out_kind_12", "idl_profiles_prepared", dict(out_kind=12), (EINVAL, "idl_profiles_prepared: float32 outputs only")),
    ("still_takes_f32", "idl_profiles_prepared", dict(out_kind=FREQ_F32, out_stride=4096), (ECUDA, CUDA)),
]


def _call_all():
    """child process: run every case, return {case key: [rc, error text]}"""
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    ws_total = lib.idl_profiles_workspace_bytes()

    def call(entry, over):
        a = dict(BASE)
        a.update(over)
        a.setdefault("n_variants", len(a["variants"]))
        a.setdefault("S", a["n_variants"])
        a.setdefault("out_off", [0] * a["S"])
        a["ws_bytes"] = ws_total
        a["prep_size"] = lib.idl_prepare_bytes(a["n_items"])
        args = []
        for name in ORDER[entry].split():
            v = a[name]
            if name == "variants":
                arr = (_lib.Variant * len(v))()
                for i, (kind, p1, p2, n_bp) in enumerate(v):
                    arr[i].kind, arr[i].rng_id, arr[i].n_bp, arr[i].explicit_idx, arr[i].p1, arr[i].p2 = kind, i, n_bp, 0, p1, p2
                v = arr
            elif name == "out_off":
                v = (ctypes.c_int64 * len(v))(*v)
            elif name in POINTERS and v is not None:
                v = ctypes.c_void_p(v)
            args.append(v)
        rc = getattr(lib, entry)(*args)
        return [rc, lib.idl_last_error().decode()]

    return {"results": {entry + "::" + cid: call(entry, over) for cid, entry, over, _ in CASES},
            "consts": [_lib.OUT_CANON_F32, _lib.OUT_CANON_STD_F32, _lib.OUT_CANON_F64]}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("case", CASES, ids=[c[1] + "::" + c[0] for c in CASES])
def test_canonical_entry_point_validation(called, case):
    cid, entry, _, (rc, text) = case
    got_rc, got_text = called["results"][entry + "::" + cid]
    assert got_rc == rc, (cid, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    else:
        assert got_text == text


def test_canonical_kind_values_match_the_header(called):
    """the Python constants are the header's enum values (8 + the matching frequency kind)"""
    txt = open(os.path.join(ROOT, "include", "idelucs_b200.h")).read()
    want = [int(re.search(r"\b%s\s*=\s*(\d+)" % n, txt).group(1)) for n in ("IDL_OUT_CANON_F32", "IDL_OUT_CANON_STD_F32", "IDL_OUT_CANON_F64")]
    assert called["consts"] == want == [CANON_F32, CANON_STD_F32, CANON_F64]


if __name__ == "__main__":
    print(json.dumps(_call_all()))
