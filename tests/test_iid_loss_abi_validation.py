"""Argument validation of the IIC loss entry points of the C ABI (idl_iid_loss, idl_iid_loss_scaled and the two sizing functions):
the return code and the exact idl_last_error() text of every argument set below.

As in test_profile_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that passes
validation fails at its first CUDA call with IDL_ECUDA instead of launching on the placeholder pointers.  The valid cases span both
sides of every size switch: the register kernel (C <= 8), the single-CTA kernel (C <= 16) and the route above 16 clusters, up to
the largest supported C.  Every output is optional, so no output, or any one of them alone, is a valid request."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, 1, 2, 3
DEV = 64   # placeholder device pointer (16-byte aligned)
ORDER = {
    "idl_iid_loss": "z1 z2 B C lamb eps loss joint dz1 dz2 ws ws_bytes stream",
    "idl_iid_loss_scaled": "z1 z2 B C lamb eps grad_scale loss_weight add add_weight loss joint dz1 dz2 ws ws_bytes stream",
}
BASE = dict(z1=DEV, z2=DEV, B=512, C=200, lamb=2.8, eps=2.2e-16, grad_scale=0.25, loss_weight=0.25, add=DEV, add_weight=0.75, loss=DEV,
            joint=DEV, dz1=DEV, dz2=DEV, ws=DEV, ws_bytes="ws", stream=None)
POINTERS = set("z1 z2 add loss joint dz1 dz2 ws stream".split())
OUTPUTS = ("loss", "joint", "dz1", "dz2")
CUDA = "<cuda>"   # any CUDA runtime error: the request got past validation

BAD = "idl_iid_loss: bad argument"
WS_SMALL = "idl_iid_loss: workspace too small"
TOO_MANY = "idl_iid_loss: n_clusters > 256 not supported (got {C})"

# (id, arguments that differ from BASE, (return code, error text or CUDA)); every case runs through both entry points
CASES = (
    [("valid_C%d" % C, dict(C=C), (ECUDA, CUDA)) for C in (1, 8, 9, 16, 17, 200, 256)]
    + [("valid_B1_C%d" % C, dict(B=1, C=C), (ECUDA, CUDA)) for C in (5, 12, 64)]
    + [("valid_large_B_C%d" % C, dict(B=100000, C=C), (ECUDA, CUDA)) for C in (8, 16, 200)]
    + [("valid_no_output_C%d" % C, dict(C=C, **{o: None for o in OUTPUTS}), (ECUDA, CUDA)) for C in (5, 12, 200)]
    + [("valid_only_%s_C%d" % (keep, C), dict(C=C, **{o: None for o in OUTPUTS if o != keep}), (ECUDA, CUDA))
       for C in (5, 12, 200) for keep in OUTPUTS]
    + [("valid_no_add", dict(add=None), (ECUDA, CUDA)),
       ("valid_workspace_larger",dict(ws_bytes="ws+1"), (ECUDA, CUDA)),
       ("null_z1", dict(z1=None), (EINVAL, BAD)),
       ("null_z2", dict(z2=None), (EINVAL, BAD)),
       ("null_workspace", dict(ws=None), (EINVAL, BAD)),
       ("null_workspace_C5", dict(C=5, ws=None), (EINVAL, BAD)),
       ("B_0", dict(B=0), (EINVAL, BAD)),
       ("B_negative", dict(B=-1), (EINVAL, BAD)),
       ("C_0", dict(C=0), (EINVAL, BAD)),
       ("C_negative", dict(C=-3), (EINVAL, BAD)),
       ("C_257", dict(C=257), (EUNSUPPORTED, TOO_MANY.format(C=257))),
       ("C_100000", dict(C=100000), (EUNSUPPORTED, TOO_MANY.format(C=100000))),
       ("C_257_null_z1", dict(C=257, z1=None), (EINVAL, BAD)),
       ("workspace_0_C17", dict(C=17, ws_bytes=0), (EINVAL, WS_SMALL))]
    + [("workspace_too_small_C%d" % C, dict(C=C, ws_bytes="ws-1"), (EINVAL, WS_SMALL)) for C in (1, 8, 16, 17, 64, 200, 256)]
)
ENTRIES = tuple(ORDER)


def _call_all():
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    out = {}
    for entry in ENTRIES:
        for cid, over, _ in CASES:
            a = dict(BASE, **over)
            ws = lib.idl_iid_loss_workspace_bytes(a["C"])
            a["ws_bytes"] = {"ws": ws, "ws-1": ws - 1, "ws+1": ws + 1}.get(a["ws_bytes"], a["ws_bytes"])
            args = [ctypes.c_void_p(a[n]) if n in POINTERS and a[n] is not None else a[n] for n in ORDER[entry].split()]
            rc = getattr(lib, entry)(*args)
            out[entry + "::" + cid] = [rc, lib.idl_last_error().decode()]
    sizes = {str(C): lib.idl_iid_loss_workspace_bytes(C) for C in [-1, 0, 257, 1 << 20] + list(range(1, 257))}
    return {"results": out, "max_clusters": lib.idl_iid_loss_max_clusters(), "workspace_bytes": sizes}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_iid_loss_entry_point_validation(called, entry, case):
    cid, _, (rc, text) = case
    key = entry + "::" + cid
    got_rc, got_text = called["results"][key]
    assert got_rc == rc, (key, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    else:
        assert got_text == text


def test_iid_loss_max_clusters(called):
    assert called["max_clusters"] == 256


def test_iid_loss_workspace_bytes(called):
    ws = {int(C): n for C, n in called["workspace_bytes"].items()}
    for C in (-1, 0, 257, 1 << 20):
        assert ws[C] == 0, C
    for C in range(1, 17):   # the single-CTA kernels need none; the size is kept for callers that allocate it
        assert ws[C] == 4 * (3 + 2 * 256 + C * C) + 64, C
    assert all(ws[C] >= 4 * C * C for C in range(1, 257)), ws
    assert all(ws[C] >= ws[C - 1] for C in range(18, 257)), ws


if __name__ == "__main__":
    print(json.dumps(_call_all()))
