"""Argument validation of the row-range entry points of the C ABI (idl_core_distances_rows, idl_silhouette_samples_rows and
idl_mreach_mst_parts): the return code and the exact idl_last_error() text of every argument set below.

As in test_hdbscan_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that
passes validation fails at its first CUDA call with IDL_ECUDA: the tables also pin where validation ends.  An empty row
range of idl_core_distances_rows makes no CUDA call at all and returns IDL_OK."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA = 0, 1, 2
DEV = 64   # placeholder device pointer
CUDA = "<cuda>"

# --- idl_core_distances_rows and idl_silhouette_samples_rows: flat argument lists
ORDER = {
    "idl_core_distances_rows": "x n D k row_begin row_end core ws ws_bytes stream",
    "idl_silhouette_samples_rows": "x labels n D n_labels row_begin row_end out ws ws_bytes stream",
}
BASE = dict(x=DEV, labels=DEV, n=1000, D=64, k=11, n_labels=10, row_begin=128, row_end=640, core=DEV, out=DEV, ws=DEV, ws_bytes="ws",
            stream=None)
POINTERS = set("x labels core out ws stream".split())

ROWS_CASES = []
for entry in ORDER:
    NULL = entry + ": null pointer"
    ROWS_CASES += [
        ("valid", entry, {}, (ECUDA, CUDA)),
        ("valid_all_rows", entry, dict(row_begin=0, row_end=1000), (ECUDA, CUDA)),
        ("valid_last_row", entry, dict(row_begin=999, row_end=1000), (ECUDA, CUDA)),
        ("valid_unaligned", entry, dict(row_begin=3, row_end=70), (ECUDA, CUDA)),
        ("null_x", entry, dict(x=None), (EINVAL, NULL)),
        ("null_workspace", entry, dict(ws=None), (EINVAL, NULL)),
        ("n0", entry, dict(n=0, row_begin=0, row_end=0), (EINVAL, entry + ": n must be in 1..2147483647 (got 0)")),
        ("D0", entry, dict(D=0), (EINVAL, entry + ": D must be >= 1 (got 0)")),
        ("begin_negative", entry, dict(row_begin=-1), (EINVAL, entry + ": row range [-1, 640) is not inside [0, 1000)")),
        ("end_above_n", entry, dict(row_end=1001), (EINVAL, entry + ": row range [128, 1001) is not inside [0, 1000)")),
        ("begin_above_end", entry, dict(row_begin=641), (EINVAL, entry + ": row range [641, 640) is not inside [0, 1000)")),
        ("begin_at_n_end_above", entry, dict(row_begin=1000, row_end=1064), (EINVAL, entry + ": row range [1000, 1064) is not inside [0, 1000)")),
        ("range_checked_before_workspace", entry, dict(row_end=2000, ws_bytes=0),
         (EINVAL, entry + ": row range [128, 2000) is not inside [0, 1000)")),
        ("workspace_too_small", entry, dict(ws_bytes="ws-1"), (EINVAL, entry + ": workspace too small (need {ws} bytes)")),
    ]
ROWS_CASES += [
    ("empty_range", "idl_core_distances_rows", dict(row_begin=500, row_end=500), (OK, None)),
    ("empty_range_at_n", "idl_core_distances_rows", dict(row_begin=1000, row_end=1000), (OK, None)),
    ("null_core", "idl_core_distances_rows", dict(core=None), (EINVAL, "idl_core_distances_rows: null pointer")),
    ("k0", "idl_core_distances_rows", dict(k=0), (EINVAL, "idl_core_distances_rows: k must be in 1..n (got 0)")),
    ("k_above_n", "idl_core_distances_rows", dict(k=1001), (EINVAL, "idl_core_distances_rows: k must be in 1..n (got 1001)")),
    ("k_checked_before_range", "idl_core_distances_rows", dict(k=0, row_begin=-5),
     (EINVAL, "idl_core_distances_rows: k must be in 1..n (got 0)")),
    # the labels are still copied and checked when the range is empty
    ("empty_range_checks_labels", "idl_silhouette_samples_rows", dict(row_begin=500, row_end=500), (ECUDA, CUDA)),
    ("null_labels", "idl_silhouette_samples_rows", dict(labels=None), (EINVAL, "idl_silhouette_samples_rows: null pointer")),
    ("null_out", "idl_silhouette_samples_rows", dict(out=None), (EINVAL, "idl_silhouette_samples_rows: null pointer")),
    ("n_labels0", "idl_silhouette_samples_rows", dict(n_labels=0), (EINVAL, "idl_silhouette_samples_rows: n_labels must be in 1..n (got 0)")),
    ("n_labels_checked_before_range", "idl_silhouette_samples_rows", dict(n_labels=1001, row_end=-1),
     (EINVAL, "idl_silhouette_samples_rows: n_labels must be in 1..n (got 1001)")),
]

# --- idl_mreach_mst_parts: host arrays of one entry per part; None stands for a null array (row_begin / row_end: None
# replaces the array built from `ranges`)
MST = "idl_mreach_mst_parts"
MNULL = MST + ": null pointer"
PBASE = dict(n_parts=2, devices=[0, 0], x=[DEV, DEV], core=[DEV, DEV], ranges=[(0, 512), (512, 1000)], row_begin=(), row_end=(), n=1000, D=64,
             src=DEV, dst=DEV, w=DEV, ws=[DEV, DEV], ws_bytes=["ws", "ws"], streams=[None, None])


def _three(**kw):
    return dict(dict(n_parts=3, devices=[0, 0, 0], x=[DEV] * 3, core=[DEV] * 3, ws=[DEV] * 3, ws_bytes=["ws"] * 3, streams=[None] * 3), **kw)


MST_CASES = [
    ("valid", {}, (ECUDA, CUDA)),
    ("valid_one_part", dict(n_parts=1, devices=[0], x=[DEV], core=[DEV], ranges=[(0, 1000)], ws=[DEV], ws_bytes=["ws"], streams=[None]),
     (ECUDA, CUDA)),
    ("valid_empty_parts", _three(ranges=[(0, 0), (0, 1000), (1000, 1000)]), (ECUDA, CUDA)),
    ("valid_distinct_devices", dict(devices=[0, 1]), (ECUDA, CUDA)),
    ("valid_extra_workspace", dict(ws_bytes=["ws+1", "ws"]), (ECUDA, CUDA)),
    ("device_out_of_range", dict(devices=[0, 99]), (ECUDA, CUDA)),   # not checked by the library: CUDA reports it
    ("n1_has_no_edges", dict(n=1, ranges=[(0, 1), (1, 1)]), (OK, None)),
    ("null_devices", dict(devices=None), (EINVAL, MNULL)),
    ("null_x_array", dict(x=None), (EINVAL, MNULL)),
    ("null_core_array", dict(core=None), (EINVAL, MNULL)),
    ("null_row_begin", dict(row_begin=None), (EINVAL, MNULL)),
    ("null_row_end", dict(row_end=None), (EINVAL, MNULL)),
    ("null_src", dict(src=None), (EINVAL, MNULL)),
    ("null_dst", dict(dst=None), (EINVAL, MNULL)),
    ("null_w", dict(w=None), (EINVAL, MNULL)),
    ("null_ws_array", dict(ws=None), (EINVAL, MNULL)),
    ("null_ws_bytes", dict(ws_bytes=None), (EINVAL, MNULL)),
    ("null_streams", dict(streams=None), (EINVAL, MNULL)),
    ("null_arrays_checked_first", dict(devices=None, n_parts=0), (EINVAL, MNULL)),
    ("null_x_of_part1", dict(x=[DEV, None]), (EINVAL, MST + ": part 1: null pointer")),
    ("null_core_of_part0", dict(core=[None, DEV]), (EINVAL, MST + ": part 0: null pointer")),
    ("null_ws_of_part2", _three(ranges=[(0, 64), (64, 128), (128, 1000)], ws=[DEV, DEV, None]), (EINVAL, MST + ": part 2: null pointer")),
    ("n_parts0", dict(n_parts=0), (EINVAL, MST + ": n_parts must be >= 1 (got 0)")),
    ("n_parts_negative", dict(n_parts=-2), (EINVAL, MST + ": n_parts must be >= 1 (got -2)")),
    ("n0", dict(n=0, ranges=[(0, 0), (0, 0)]), (EINVAL, MST + ": n must be in 1..2147483647 (got 0)")),
    ("D0", dict(D=0), (EINVAL, MST + ": D must be >= 1 (got 0)")),
    ("begin_negative", dict(ranges=[(-1, 512), (512, 1000)]), (EINVAL, MST + ": part 0: row range [-1, 512) is not inside [0, 1000)")),
    ("end_above_n", dict(ranges=[(0, 512), (512, 1001)]), (EINVAL, MST + ": part 1: row range [512, 1001) is not inside [0, 1000)")),
    ("begin_above_end", _three(ranges=[(0, 600), (600, 400), (400, 1000)]),
     (EINVAL, MST + ": part 1: row range [600, 400) is not inside [0, 1000)")),
    ("gap", dict(ranges=[(0, 500), (501, 1000)]), (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 1 begins at 501, not 500")),
    ("overlap", dict(ranges=[(0, 500), (400, 1000)]),
     (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 1 begins at 400, not 500")),
    ("not_from_0", dict(ranges=[(64, 512), (512, 1000)]),
     (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 0 begins at 64, not 0")),
    ("short_of_n", dict(ranges=[(0, 512), (512, 900)]),
     (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 1 ends at 900, not 1000")),
    ("out_of_order", dict(ranges=[(512, 1000), (0, 512)]),
     (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 0 begins at 512, not 0")),
    ("same_range_twice", dict(ranges=[(0, 1000), (0, 1000)]),
     (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 1 begins at 0, not 1000")),
    ("range_checked_before_partition", dict(ranges=[(64, 512), (512, 2000)]),
     (EINVAL, MST + ": part 1: row range [512, 2000) is not inside [0, 1000)")),
    ("partition_checked_before_workspace", dict(ranges=[(0, 500), (501, 1000)], ws_bytes=[0, 0]),
     (EINVAL, MST + ": the row ranges do not partition [0, 1000) in order: part 1 begins at 501, not 500")),
    ("workspace_too_small_part1", dict(ws_bytes=["ws", "ws-1"]), (EINVAL, MST + ": part 1: workspace too small (need {ws} bytes)")),
    ("workspace_0_part0", dict(ws_bytes=[0, "ws"]), (EINVAL, MST + ": part 0: workspace too small (need {ws} bytes)")),
    ("empty_part_still_needs_workspace", _three(ranges=[(0, 0), (0, 1000), (1000, 1000)], ws_bytes=["ws", "ws", 0]),
     (EINVAL, MST + ": part 2: workspace too small (need {ws} bytes)")),
]


def _call_all():
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    out, wss = {}, {}
    for cid, entry, over, _ in ROWS_CASES:
        a = dict(BASE, **over)
        need = (lib.idl_hdbscan_workspace_bytes(a["n"], a["D"]) if entry == "idl_core_distances_rows"
                else lib.idl_silhouette_workspace_bytes(a["n"], a["n_labels"]))
        a["ws_bytes"] = {"ws": need, "ws-1": need - 1}.get(a["ws_bytes"], a["ws_bytes"])
        args = [ctypes.c_void_p(a[k]) if k in POINTERS and a[k] is not None else a[k] for k in ORDER[entry].split()]
        rc = getattr(lib, entry)(*args)
        out[entry + "::" + cid] = [rc, lib.idl_last_error().decode()]
        wss[entry + "::" + cid] = need
    for cid, over, _ in MST_CASES:
        a = dict(PBASE, **over)
        need = lib.idl_hdbscan_workspace_bytes(a["n"], a["D"])

        def arr(ctype, values):
            return None if values is None else (ctype * len(values))(*values)

        def one(v):
            return None if v is None else ctypes.c_void_p(v)
        begin = None if a["row_begin"] is None else [b for b, _ in a["ranges"]]
        end = None if a["row_end"] is None else [e for _, e in a["ranges"]]
        ws_bytes = None if a["ws_bytes"] is None else [{"ws": need, "ws-1": need - 1, "ws+1": need + 1}.get(b, b) for b in a["ws_bytes"]]
        rc = lib.idl_mreach_mst_parts(a["n_parts"], arr(ctypes.c_int, a["devices"]), arr(ctypes.c_void_p, a["x"]), arr(ctypes.c_void_p, a["core"]),
                                      arr(ctypes.c_int64, begin), arr(ctypes.c_int64, end), a["n"], a["D"], one(a["src"]), one(a["dst"]),
                                      one(a["w"]), arr(ctypes.c_void_p, a["ws"]), arr(ctypes.c_size_t, ws_bytes), arr(ctypes.c_void_p, a["streams"]))
        out[MST + "::" + cid] = [rc, lib.idl_last_error().decode()]
        wss[MST + "::" + cid] = need
    return {"results": out, "ws": wss}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


def _check(called, key, rc, text):
    got_rc, got_text = called["results"][key]
    assert got_rc == rc, (key, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    elif text is not None:
        assert got_text == text.format(ws=called["ws"][key])


@pytest.mark.parametrize("case", ROWS_CASES, ids=[c[1] + "::" + c[0] for c in ROWS_CASES])
def test_rows_entry_point_validation(called, case):
    cid, entry, _, (rc, text) = case
    _check(called, entry + "::" + cid, rc, text)


@pytest.mark.parametrize("case", MST_CASES, ids=[c[0] for c in MST_CASES])
def test_mreach_mst_parts_validation(called, case):
    cid, _, (rc, text) = case
    _check(called, MST + "::" + cid, rc, text)


if __name__ == "__main__":
    print(json.dumps(_call_all()))
