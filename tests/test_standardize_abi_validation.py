"""Argument validation of idl_standardize_f32 and idl_standardize_f64: the return code and the exact idl_last_error()
text of every argument set below.

As in test_profile_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that
passes validation fails at its first CUDA call with IDL_ECUDA: the tables also pin where validation ends.  In particular
idl_standardize_f32 takes any width F >= 1, not only multiples of 4: the canonical k-mer profiles of k = 1 and 2
(--model_size small) are R = 2 and R = 10 columns wide."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA = 0, 1, 2
DEV = 64   # placeholder device pointer (16-byte aligned)
ORDER = {
    "idl_standardize_f32": "x out n F mean scale stream",
    "idl_standardize_f64": "x out64 out32 n F mean scale stream",
}
BASE = dict(x=DEV, out=DEV, out64=DEV, out32=None, n=1000, F=4096, mean=DEV, scale=DEV, stream=None)
POINTERS = set("x out out64 out32 mean scale stream".split())
CUDA = "<cuda>"
BAD32 = "idl_standardize_f32: bad argument"
BAD64 = "idl_standardize_f64: bad argument"

CASES = [
    ("valid_F4096", "idl_standardize_f32", {}, (ECUDA, CUDA)),
    ("valid_F12", "idl_standardize_f32", dict(F=12), (ECUDA, CUDA)),
    ("valid_F1", "idl_standardize_f32", dict(F=1), (ECUDA, CUDA)),
    ("valid_F2", "idl_standardize_f32", dict(F=2), (ECUDA, CUDA)),
    ("valid_F10", "idl_standardize_f32", dict(F=10), (ECUDA, CUDA)),
    ("valid_F2080", "idl_standardize_f32", dict(F=2080), (ECUDA, CUDA)),
    ("n0", "idl_standardize_f32", dict(n=0, F=10), (OK, None)),
    ("F0", "idl_standardize_f32", dict(F=0), (EINVAL, BAD32)),
    ("F_negative", "idl_standardize_f32", dict(F=-2), (EINVAL, BAD32)),
    ("n_negative", "idl_standardize_f32", dict(n=-1), (EINVAL, BAD32)),
    ("n_negative_F10", "idl_standardize_f32", dict(n=-1, F=10), (EINVAL, BAD32)),
    ("null_x", "idl_standardize_f32", dict(x=None), (EINVAL, BAD32)),
    ("null_out", "idl_standardize_f32", dict(out=None), (EINVAL, BAD32)),
    ("null_mean", "idl_standardize_f32", dict(mean=None), (EINVAL, BAD32)),
    ("null_scale", "idl_standardize_f32", dict(scale=None), (EINVAL, BAD32)),
    ("null_x_F2", "idl_standardize_f32", dict(x=None, F=2), (EINVAL, BAD32)),
    ("null_scale_F10", "idl_standardize_f32", dict(scale=None, F=10), (EINVAL, BAD32)),
    ("null_checked_when_n0", "idl_standardize_f32", dict(n=0, mean=None), (EINVAL, BAD32)),

    ("valid_F10", "idl_standardize_f64", dict(F=10), (ECUDA, CUDA)),
    ("valid_out32_only", "idl_standardize_f64", dict(out64=None, out32=DEV, F=2), (ECUDA, CUDA)),
    ("n0", "idl_standardize_f64", dict(n=0), (OK, None)),
    ("no_output", "idl_standardize_f64", dict(out64=None), (EINVAL, BAD64)),
    ("F0", "idl_standardize_f64", dict(F=0), (EINVAL, BAD64)),
    ("n_negative", "idl_standardize_f64", dict(n=-1), (EINVAL, BAD64)),
    ("null_mean", "idl_standardize_f64", dict(mean=None), (EINVAL, BAD64)),
]


def _call_all():
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    out = {}
    for cid, entry, over, _ in CASES:
        a = dict(BASE, **over)
        args = [ctypes.c_void_p(a[k]) if k in POINTERS and a[k] is not None else a[k] for k in ORDER[entry].split()]
        rc = getattr(lib, entry)(*args)
        out[entry + "::" + cid] = [rc, lib.idl_last_error().decode()]
    return {"results": out}


@pytest.fixture(scope="module")
def called():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("case", CASES, ids=[c[1] + "::" + c[0] for c in CASES])
def test_standardize_entry_point_validation(called, case):
    cid, entry, _, (rc, text) = case
    key = entry + "::" + cid
    got_rc, got_text = called["results"][key]
    assert got_rc == rc, (key, got_rc, got_text)
    if text == CUDA:
        assert re.fullmatch(r".+ \(cuda error \d+\)", got_text), got_text
    elif text is not None:
        assert got_text == text


if __name__ == "__main__":
    print(json.dumps(_call_all()))
