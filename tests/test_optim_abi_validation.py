"""Argument validation of the SGD and Adam entry points of the C ABI (idl_sgd_step, idl_adam_step and their *_allreduce_step
variants): the return code and the exact idl_last_error() text of every argument set below.

As in test_train_ops_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that passes
validation fails at its first CUDA call with IDL_ECUDA instead of launching on the placeholder pointers: a missing check shows up
as a CUDA error here, never as a fault.  The step counter is an int64 the kernels read, so it must be 8-byte aligned; the
all-reduce kernels access their buffers as float4, so their state buffers, peer pointers and multicast addresses must be 16-byte
aligned."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL = 0, 1
ECUDA = 2
DEV = 64    # placeholder device pointer (16-byte aligned)
ODD = 68    # placeholder device pointer, 4-byte aligned only
ORDER = {
    "idl_sgd_step": "param grad buf n lr momentum wd step grad_scale stream",
    "idl_adam_step": "param grad m v n lr beta1 beta2 eps wd step grad_scale stream",
    "idl_sgd_allreduce_step": "grad_peers param_peers grad_mc param_mc buf n_total rank world lr momentum wd step stream",
    "idl_adam_allreduce_step": "grad_peers param_peers grad_mc param_mc m v n_total rank world lr beta1 beta2 eps wd step stream",
}
BASE = dict(param=DEV, grad=DEV, buf=DEV, m=DEV, v=DEV, n=4096, lr=1e-3, momentum=0.9, wd=0.01, beta1=0.9, beta2=0.999, eps=1e-8,
            step=DEV, grad_scale=0.5, grad_peers="world", param_peers="world", grad_mc=0, param_mc=0, n_total=1024, rank=0, world=2,
            stream=None)
POINTERS = set("param grad buf m v step stream".split())
CUDA = "<cuda>"   # any CUDA runtime error: the request got past validation

SGD = "idl_sgd_step: bad argument"
SGD_STEP = "idl_sgd_step: null / misaligned step counter (int64 in device memory)"
ADAM = "idl_adam_step: bad argument"
ADAM_STEP = "idl_adam_step: null / misaligned step counter (int64 in device memory)"


def _ar(name):
    return dict(bad="%s: bad argument (n_total must be a multiple of 4 x world, world <= 16)" % name,
                peer="%s: null / misaligned peer pointer" % name,
                step="%s: null / misaligned step counter (int64 in device memory)" % name)


SAR, AAR = _ar("idl_sgd_allreduce_step"), _ar("idl_adam_allreduce_step")
SAR["align"] = "idl_sgd_allreduce_step: misaligned momentum_buffer / multicast address"
AAR["align"] = "idl_adam_allreduce_step: misaligned exp_avg / exp_avg_sq / multicast address"


def _peers(world, **at):
    """placeholder peer table of `world` ranks (distinct aligned addresses); at = {rank: address} overrides"""
    return [at.get("r%d" % r, DEV * (r + 1)) for r in range(world)]


# (id, entry point, arguments that differ from BASE, (return code, error text or CUDA or None))
CASES = [
    ("valid", "idl_sgd_step", {}, (ECUDA, CUDA)),
    ("valid_unaligned_buffers", "idl_sgd_step", dict(param=ODD, grad=ODD, buf=ODD, n=5), (ECUDA, CUDA)),
    ("valid_step_8_aligned", "idl_sgd_step", dict(step=DEV + 8), (ECUDA, CUDA)),
    ("n_0", "idl_sgd_step", dict(n=0), (OK, None)),
    ("null_param", "idl_sgd_step", dict(param=None), (EINVAL, SGD)),
    ("null_grad", "idl_sgd_step", dict(grad=None), (EINVAL, SGD)),
    ("null_momentum_buffer", "idl_sgd_step", dict(buf=None), (EINVAL, SGD)),
    ("n_negative", "idl_sgd_step", dict(n=-1), (EINVAL, SGD)),
    ("null_step", "idl_sgd_step", dict(step=None), (EINVAL, SGD_STEP)),
    ("misaligned_step", "idl_sgd_step", dict(step=ODD), (EINVAL, SGD_STEP)),
    ("null_step_checked_when_n_0", "idl_sgd_step", dict(n=0, step=None), (EINVAL, SGD_STEP)),

    ("valid", "idl_adam_step", {}, (ECUDA, CUDA)),
    ("valid_unaligned_buffers", "idl_adam_step", dict(param=ODD, grad=ODD, m=ODD, v=ODD, n=7), (ECUDA, CUDA)),
    ("n_0", "idl_adam_step", dict(n=0), (OK, None)),
    ("null_param", "idl_adam_step", dict(param=None), (EINVAL, ADAM)),
    ("null_grad", "idl_adam_step", dict(grad=None), (EINVAL, ADAM)),
    ("null_exp_avg", "idl_adam_step", dict(m=None), (EINVAL, ADAM)),
    ("null_exp_avg_sq", "idl_adam_step", dict(v=None), (EINVAL, ADAM)),
    ("n_negative", "idl_adam_step", dict(n=-4), (EINVAL, ADAM)),
    ("null_step", "idl_adam_step", dict(step=None), (EINVAL, ADAM_STEP)),
    ("misaligned_step", "idl_adam_step", dict(step=DEV + 4), (EINVAL, ADAM_STEP)),
]
for entry, E, state in (("idl_sgd_allreduce_step", SAR, ("buf",)), ("idl_adam_allreduce_step", AAR, ("m", "v"))):
    CASES += [
        ("valid", entry, {}, (ECUDA, CUDA)),
        ("valid_world_1", entry, dict(world=1, n_total=4), (ECUDA, CUDA)),
        ("valid_world_16_last_rank", entry, dict(world=16, rank=15, n_total=64), (ECUDA, CUDA)),
        ("valid_multicast", entry, dict(grad_mc=1 << 40, param_mc=(1 << 40) + 4096), (ECUDA, CUDA)),
        ("world_17", entry, dict(world=17, n_total=17 * 64), (EINVAL, E["bad"])),
        ("world_0", entry, dict(world=0), (EINVAL, E["bad"])),
        ("rank_negative", entry, dict(rank=-1), (EINVAL, E["bad"])),
        ("rank_equals_world", entry, dict(rank=2), (EINVAL, E["bad"])),
        ("n_total_0", entry, dict(n_total=0), (EINVAL, E["bad"])),
        ("n_total_negative", entry, dict(n_total=-8), (EINVAL, E["bad"])),
        ("n_total_not_multiple_of_4_world", entry, dict(n_total=1028), (EINVAL, E["bad"])),
        ("n_total_3_world", entry, dict(world=3, n_total=3 * 4 * 5 + 4), (EINVAL, E["bad"])),
        ("null_grad_table", entry, dict(grad_peers=None), (EINVAL, E["bad"])),
        ("null_param_table", entry, dict(param_peers=None), (EINVAL, E["bad"])),
        ("null_grad_peer", entry, dict(grad_peers=dict(r1=0)), (EINVAL, E["peer"])),
        ("null_param_peer", entry, dict(param_peers=dict(r0=0)), (EINVAL, E["peer"])),
        ("misaligned_grad_peer", entry, dict(grad_peers=dict(r1=ODD)), (EINVAL, E["peer"])),
        ("misaligned_param_peer", entry, dict(param_peers=dict(r0=DEV + 8)), (EINVAL, E["peer"])),
        ("misaligned_grad_multicast", entry, dict(grad_mc=(1 << 40) + 4, param_mc=1 << 40), (EINVAL, E["align"])),
        ("misaligned_param_multicast", entry, dict(grad_mc=1 << 40, param_mc=(1 << 40) + 8), (EINVAL, E["align"])),
        ("null_step", entry, dict(step=None), (EINVAL, E["step"])),
        ("misaligned_step", entry, dict(step=DEV + 4), (EINVAL, E["step"])),
    ]
    for s in state:
        CASES += [
            ("null_" + s, entry, {s: None}, (EINVAL, E["bad"])),
            ("misaligned_" + s, entry, {s: ODD}, (EINVAL, E["align"])),
            ("misaligned_8_" + s, entry, {s: DEV + 8}, (EINVAL, E["align"])),
        ]


def _call_all():
    import ctypes
    sys.path.insert(0, ROOT)
    from idelucs_b200 import _lib
    lib = _lib.load()
    out = {}
    for cid, entry, over, _ in CASES:
        a = dict(BASE, **over)
        args = []
        for name in ORDER[entry].split():
            v = a[name]
            if name in ("grad_peers", "param_peers") and v is not None:
                table = _peers(a["world"], **(v if isinstance(v, dict) else {}))
                v = (ctypes.c_uint64 * len(table))(*table)
            elif name in POINTERS and v is not None:
                v = ctypes.c_void_p(v)
            args.append(v)
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
def test_optimizer_entry_point_validation(called, case):
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
