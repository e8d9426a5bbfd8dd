"""Argument validation of the silhouette entry points of the C ABI (idl_silhouette_samples and
idl_silhouette_workspace_bytes): the return code and the exact idl_last_error() text of every argument set below.

As in test_hdbscan_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that
passes validation fails at its first CUDA call (the copy of the labels to the host) with IDL_ECUDA: the table also pins
where validation ends."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA = 0, 1, 2
DEV = 64   # placeholder device pointer
ENTRY = "idl_silhouette_samples"
ORDER = "x labels n D n_labels out ws ws_bytes stream".split()
BASE = dict(x=DEV, labels=DEV, n=1000, D=64, n_labels=10, out=DEV, ws=DEV, ws_bytes="ws", stream=None)
POINTERS = set("x labels out ws stream".split())
CUDA = "<cuda>"
NULL = ENTRY + ": null pointer"

CASES = [
    ("valid", {}, (ECUDA, CUDA)),
    ("valid_D1", dict(D=1), (ECUDA, CUDA)),
    ("valid_n1", dict(n=1, n_labels=1), (ECUDA, CUDA)),
    ("valid_one_label", dict(n_labels=1), (ECUDA, CUDA)),
    ("valid_n_labels_n", dict(n_labels=1000), (ECUDA, CUDA)),
    ("valid_extra_workspace", dict(ws_bytes="ws+1"), (ECUDA, CUDA)),
    ("null_x", dict(x=None), (EINVAL, NULL)),
    ("null_labels", dict(labels=None), (EINVAL, NULL)),
    ("null_out", dict(out=None), (EINVAL, NULL)),
    ("null_workspace", dict(ws=None), (EINVAL, NULL)),
    ("null_checked_first", dict(x=None, n=0, D=0, ws_bytes=0), (EINVAL, NULL)),
    ("n0", dict(n=0), (EINVAL, ENTRY + ": n must be in 1..2147483647 (got 0)")),
    ("n_negative", dict(n=-4), (EINVAL, ENTRY + ": n must be in 1..2147483647 (got -4)")),
    ("n_2_31", dict(n=2 ** 31, ws_bytes=1 << 40), (EINVAL, ENTRY + ": n must be in 1..2147483647 (got 2147483648)")),
    ("D0", dict(D=0), (EINVAL, ENTRY + ": D must be >= 1 (got 0)")),
    ("D_negative", dict(D=-3), (EINVAL, ENTRY + ": D must be >= 1 (got -3)")),
    ("n_labels0", dict(n_labels=0), (EINVAL, ENTRY + ": n_labels must be in 1..n (got 0)")),
    ("n_labels_negative", dict(n_labels=-2), (EINVAL, ENTRY + ": n_labels must be in 1..n (got -2)")),
    ("n_labels_above_n", dict(n_labels=1001), (EINVAL, ENTRY + ": n_labels must be in 1..n (got 1001)")),
    ("n_labels_checked_before_workspace", dict(n_labels=0, ws_bytes=0), (EINVAL, ENTRY + ": n_labels must be in 1..n (got 0)")),
    ("workspace_too_small", dict(ws_bytes="ws-1"), (EINVAL, ENTRY + ": workspace too small (need {ws} bytes)")),
    ("workspace_0", dict(ws_bytes=0), (EINVAL, ENTRY + ": workspace too small (need {ws} bytes)")),
]

# idl_silhouette_workspace_bytes: (id, n, n_labels, expected: 0 or "positive")
SIZES = [("n0", 0, 1, 0), ("n_negative", -1, 1, 0), ("n_2_31", 2 ** 31, 2, 0), ("n_labels0", 10, 0, 0), ("n_labels_negative", 10, -1, 0),
         ("n_labels_above_n", 10, 11, 0), ("n1", 1, 1, "positive"), ("n_labels_n", 10, 10, "positive"), ("n_max", 2 ** 31 - 1, 2, "positive")]


def _call_all():
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    out, ws = {}, {}
    for cid, over, _ in CASES:
        a = dict(BASE, **over)
        need = lib.idl_silhouette_workspace_bytes(a["n"], a["n_labels"])
        a["ws_bytes"] = {"ws": need, "ws-1": need - 1, "ws+1": need + 1}.get(a["ws_bytes"], a["ws_bytes"])
        args = [ctypes.c_void_p(a[k]) if k in POINTERS and a[k] is not None else a[k] for k in ORDER]
        rc = lib.idl_silhouette_samples(*args)
        out[cid] = [rc, lib.idl_last_error().decode()]
        ws[cid] = need
    sizes = {cid: lib.idl_silhouette_workspace_bytes(n, m) for cid, n, m, _ in SIZES}
    grow = [lib.idl_silhouette_workspace_bytes(n, 2) for n in (1000, 10 ** 6, 10 ** 8)]
    by_labels = [lib.idl_silhouette_workspace_bytes(10 ** 6, m) for m in (2, 10 ** 6)]
    return {"results": out, "ws": ws, "sizes": sizes, "grow": grow, "by_labels": by_labels}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_silhouette_entry_point_validation(called, case):
    cid, _, (rc, text) = case
    got_rc, got_text = called["results"][cid]
    assert got_rc == rc, (cid, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    else:
        assert got_text == text.format(ws=called["ws"][cid])


@pytest.mark.parametrize("case", SIZES, ids=[c[0] for c in SIZES])
def test_silhouette_workspace_bytes(called, case):
    cid, _, _, want = case
    got = called["sizes"][cid]
    assert got > 0 if want == "positive" else got == want


def test_silhouette_workspace_is_linear_in_n(called):
    """int32 order [n] + int32 offsets [n_labels + 1]: about 4 bytes per point and per label, no n x n buffer"""
    a, b, c = called["grow"]
    assert 0 < a < b < c and 4 * 10 ** 8 <= c <= 4 * 10 ** 8 + 1024
    few, many = called["by_labels"]
    assert 4 * 10 ** 6 <= few <= 4 * 10 ** 6 + 1024 and 8 * 10 ** 6 <= many <= 8 * 10 ** 6 + 1024


if __name__ == "__main__":
    print(json.dumps(_call_all()))
