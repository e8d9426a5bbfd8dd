"""Argument validation of the HDBSCAN entry points of the C ABI (idl_core_distances, idl_mreach_mst and
idl_hdbscan_workspace_bytes): the return code and the exact idl_last_error() text of every argument set below.

As in test_profile_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that
passes validation fails at its first CUDA call with IDL_ECUDA: the tables also pin where validation ends."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA = 0, 1, 2
DEV = 64   # placeholder device pointer
ORDER = {
    "idl_core_distances": "x n D k core ws ws_bytes stream",
    "idl_mreach_mst": "x core n D src dst w ws ws_bytes stream",
}
BASE = dict(x=DEV, n=1000, D=64, k=11, core=DEV, src=DEV, dst=DEV, w=DEV, ws=DEV, ws_bytes="ws", stream=None)
POINTERS = set("x core src dst w ws stream".split())
CUDA = "<cuda>"

CASES = []
for entry in ORDER:
    NULL = entry + ": null pointer"
    CASES += [
        ("valid", entry, {}, (ECUDA, CUDA)),
        ("valid_D1", entry, dict(D=1), (ECUDA, CUDA)),
        ("null_x", entry, dict(x=None), (EINVAL, NULL)),
        ("null_core", entry, dict(core=None), (EINVAL, NULL)),
        ("null_workspace", entry, dict(ws=None), (EINVAL, NULL)),
        ("n0", entry, dict(n=0), (EINVAL, entry + ": n must be in 1..2147483647 (got 0)")),
        ("n_negative", entry, dict(n=-4), (EINVAL, entry + ": n must be in 1..2147483647 (got -4)")),
        ("n_2_31", entry, dict(n=2 ** 31, ws_bytes=1 << 40), (EINVAL, entry + ": n must be in 1..2147483647 (got 2147483648)")),
        ("D0", entry, dict(D=0), (EINVAL, entry + ": D must be >= 1 (got 0)")),
        ("D_negative", entry, dict(D=-3), (EINVAL, entry + ": D must be >= 1 (got -3)")),
        ("workspace_too_small", entry, dict(ws_bytes="ws-1"), (EINVAL, entry + ": workspace too small (need {ws} bytes)")),
        ("workspace_0", entry, dict(ws_bytes=0), (EINVAL, entry + ": workspace too small (need {ws} bytes)")),
    ]
CASES += [
    ("valid_k1", "idl_core_distances", dict(k=1), (ECUDA, CUDA)),
    ("valid_k_n", "idl_core_distances", dict(k=1000), (ECUDA, CUDA)),
    ("valid_n1", "idl_core_distances", dict(n=1, k=1), (ECUDA, CUDA)),
    ("k0", "idl_core_distances", dict(k=0), (EINVAL, "idl_core_distances: k must be in 1..n (got 0)")),
    ("k_negative", "idl_core_distances", dict(k=-1), (EINVAL, "idl_core_distances: k must be in 1..n (got -1)")),
    ("k_above_n", "idl_core_distances", dict(k=1001), (EINVAL, "idl_core_distances: k must be in 1..n (got 1001)")),
    ("k_checked_before_workspace", "idl_core_distances", dict(k=0, ws_bytes=0), (EINVAL, "idl_core_distances: k must be in 1..n (got 0)")),
    ("null_src", "idl_mreach_mst", dict(src=None), (EINVAL, "idl_mreach_mst: null pointer")),
    ("null_dst", "idl_mreach_mst", dict(dst=None), (EINVAL, "idl_mreach_mst: null pointer")),
    ("null_w", "idl_mreach_mst", dict(w=None), (EINVAL, "idl_mreach_mst: null pointer")),
    ("n1_has_no_edges", "idl_mreach_mst", dict(n=1), (OK, None)),
]

# idl_hdbscan_workspace_bytes: (id, n, D, expected: 0 or "positive")
SIZES = [("n0", 0, 64, 0), ("n_negative", -1, 64, 0), ("D0", 10, 0, 0), ("n_2_31", 2 ** 31, 64, 0),
         ("n1", 1, 1, "positive"), ("n_max", 2 ** 31 - 1, 64, "positive")]


def _call_all():
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    out, ws = {}, {}
    for cid, entry, over, _ in CASES:
        a = dict(BASE, **over)
        need = lib.idl_hdbscan_workspace_bytes(a["n"], a["D"])
        a["ws_bytes"] = {"ws": need, "ws-1": need - 1}.get(a["ws_bytes"], a["ws_bytes"])
        args = [ctypes.c_void_p(a[k]) if k in POINTERS and a[k] is not None else a[k] for k in ORDER[entry].split()]
        rc = getattr(lib, entry)(*args)
        out[entry + "::" + cid] = [rc, lib.idl_last_error().decode()]
        ws[entry + "::" + cid] = need
    sizes = {cid: lib.idl_hdbscan_workspace_bytes(n, D) for cid, n, D, _ in SIZES}
    grow = [lib.idl_hdbscan_workspace_bytes(n, 64) for n in (1, 1000, 10 ** 6)]
    return {"results": out, "ws": ws, "sizes": sizes, "grow": grow}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("case", CASES, ids=[c[1] + "::" + c[0] for c in CASES])
def test_hdbscan_entry_point_validation(called, case):
    cid, entry, _, (rc, text) = case
    key = entry + "::" + cid
    got_rc, got_text = called["results"][key]
    assert got_rc == rc, (key, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    elif text is not None:
        assert got_text == text.format(ws=called["ws"][key])


@pytest.mark.parametrize("case", SIZES, ids=[c[0] for c in SIZES])
def test_hdbscan_workspace_bytes(called, case):
    cid, _, _, want = case
    got = called["sizes"][cid]
    assert got > 0 if want == "positive" else got == want


def test_hdbscan_workspace_is_linear_in_n(called):
    a, b, c = called["grow"]
    assert 0 < a < b < c and c <= 64 * 10 ** 6   # O(n) bytes: no n x n buffer


if __name__ == "__main__":
    print(json.dumps(_call_all()))
