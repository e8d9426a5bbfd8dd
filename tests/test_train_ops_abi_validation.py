"""Argument validation of the training-step entry points of the C ABI (the InfoNCE pieces, the fused ReLU - Dropout kernels,
idl_sum_parts_bias, idl_pair_selection and the two RMSprop steps): the return code and the exact idl_last_error() text of every
argument set below.

As in test_profile_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that passes
validation fails at its first CUDA call with IDL_ECUDA instead of launching on the placeholder pointers: a missing check shows up
as a CUDA error here, never as a fault.  The kernels behind idl_relu_dropout_forward / _backward, idl_sum_parts_bias and
idl_rmsprop_allreduce_step access their buffers as float4, so a buffer that is not 16-byte aligned (a torch view at an odd storage
offset) is rejected; idl_nce_softmax_xent takes the scalar weights kernel for such a buffer instead."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA = 0, 1, 2
DEV = 64    # placeholder device pointer (16-byte aligned)
ODD = 68    # placeholder device pointer, 4-byte aligned only
NAN = float("nan")
ORDER = {
    "idl_nce_normalize": "h n2 D fn inv_norm stream",
    "idl_nce_softmax_xent": "sim n2 temperature lse rowloss loss stream",
    "idl_nce_softmax_xent_scaled": "sim n2 temperature grad_scale lse rowloss loss stream",
    "idl_nce_normalize_backward": "dfn fn inv_norm n2 D dh stream",
    "idl_nce_normalize_backward_parts": "dfn n_parts fn inv_norm n2 D dh stream",
    "idl_relu_dropout_forward": "parts n_parts bias M N p seed step tag out stream",
    "idl_relu_dropout_backward": "out dy n p dx stream",
    "idl_sum_parts_bias": "parts n_parts bias M N out stream",
    "idl_pair_selection": "pair_ids n_pairs n_seqs sidx sel stream",
    "idl_rmsprop_step": "param grad sq n lr alpha eps wd grad_scale stream",
    "idl_rmsprop_allreduce_step": "grad_peers param_peers grad_mc param_mc sq n_total rank world lr alpha eps wd stream",
}
BASE = dict(h=DEV, n2=1024, D=64, fn=DEV, inv_norm=DEV, sim=DEV, temperature=0.85, grad_scale=0.75, lse=DEV, rowloss=DEV, loss=DEV,
            dfn=DEV, n_parts=4, dh=DEV, parts=DEV, bias=DEV, M=1024, N=512, p=0.5, seed=(1 << 40) + 7, step=DEV, tag=1, out=DEV,
            dy=DEV, n=4096, dx=DEV, pair_ids=DEV, n_pairs=512, n_seqs=1000, sidx=DEV, sel=DEV, param=DEV, grad=DEV, sq=DEV, lr=1e-3,
            alpha=0.99, eps=1e-8, wd=0.01, grad_peers="world", param_peers="world", grad_mc=0, param_mc=0, n_total=1024, rank=0,
            world=2, stream=None)
POINTERS = set("h fn inv_norm sim lse rowloss loss dfn dh parts bias step out dy dx pair_ids sidx sel param grad sq stream".split())
CUDA = "<cuda>"   # any CUDA runtime error: the request got past validation

NORM = "idl_nce_normalize: bad argument"
XENT = "idl_nce_softmax_xent: bad argument"
NBWD = "idl_nce_normalize_backward: bad argument"
FWD = "idl_relu_dropout_forward: bad argument (N must be a multiple of 4, 0 <= p < 1)"
FWD_ALIGN = "idl_relu_dropout_forward: misaligned buffer (parts, bias and out are read and written as float4)"
BWD = "idl_relu_dropout_backward: bad argument"
BWD_ALIGN = "idl_relu_dropout_backward: misaligned buffer (out, dy and dx are read and written as float4)"
SUM = "idl_sum_parts_bias: bad argument (N must be a multiple of 4)"
SUM_ALIGN = "idl_sum_parts_bias: misaligned buffer (parts, bias and out are read and written as float4)"
PAIR = "idl_pair_selection: bad argument"
RMS = "idl_rmsprop_step: bad argument"
AR = "idl_rmsprop_allreduce_step: bad argument (n_total must be a multiple of 4 x world, world <= 16)"
AR_PEER = "idl_rmsprop_allreduce_step: null / misaligned peer pointer"
AR_ALIGN = "idl_rmsprop_allreduce_step: misaligned square_avg / multicast address"


def _peers(world, **at):
    """placeholder peer table of `world` ranks (distinct aligned addresses); at = {rank: address} overrides"""
    return [at.get("r%d" % r, DEV * (r + 1)) for r in range(world)]


# (id, entry point, arguments that differ from BASE, (return code, error text or CUDA or None))
CASES = [
    ("valid", "idl_nce_normalize", {}, (ECUDA, CUDA)),
    ("valid_one_row_odd_D", "idl_nce_normalize", dict(n2=1, D=3, h=ODD, fn=ODD), (ECUDA, CUDA)),
    ("null_h", "idl_nce_normalize", dict(h=None), (EINVAL, NORM)),
    ("null_fn", "idl_nce_normalize", dict(fn=None), (EINVAL, NORM)),
    ("null_inv_norm", "idl_nce_normalize", dict(inv_norm=None), (EINVAL, NORM)),
    ("n2_0", "idl_nce_normalize", dict(n2=0), (EINVAL, NORM)),
    ("D_0", "idl_nce_normalize", dict(D=0), (EINVAL, NORM)),

    ("valid", "idl_nce_softmax_xent", {}, (ECUDA, CUDA)),
    ("valid_without_loss", "idl_nce_softmax_xent", dict(loss=None), (ECUDA, CUDA)),
    ("valid_n2_2", "idl_nce_softmax_xent", dict(n2=2), (ECUDA, CUDA)),
    ("valid_n2_666_scalar_kernel", "idl_nce_softmax_xent", dict(n2=666), (ECUDA, CUDA)),
    ("misaligned_sim_takes_scalar_kernel", "idl_nce_softmax_xent", dict(sim=ODD), (ECUDA, CUDA)),
    ("misaligned_lse_takes_scalar_kernel", "idl_nce_softmax_xent", dict(lse=ODD), (ECUDA, CUDA)),
    ("null_sim", "idl_nce_softmax_xent", dict(sim=None), (EINVAL, XENT)),
    ("null_lse", "idl_nce_softmax_xent", dict(lse=None), (EINVAL, XENT)),
    ("null_rowloss", "idl_nce_softmax_xent", dict(rowloss=None), (EINVAL, XENT)),
    ("n2_0", "idl_nce_softmax_xent", dict(n2=0), (EINVAL, XENT)),
    ("n2_odd", "idl_nce_softmax_xent", dict(n2=1023), (EINVAL, XENT)),
    ("temperature_0", "idl_nce_softmax_xent", dict(temperature=0.0), (EINVAL, XENT)),
    ("temperature_negative", "idl_nce_softmax_xent", dict(temperature=-0.85), (EINVAL, XENT)),
    ("temperature_nan", "idl_nce_softmax_xent", dict(temperature=NAN), (EINVAL, XENT)),
    ("valid", "idl_nce_softmax_xent_scaled", {}, (ECUDA, CUDA)),
    ("valid_grad_scale_0", "idl_nce_softmax_xent_scaled", dict(grad_scale=0.0), (ECUDA, CUDA)),
    ("null_sim", "idl_nce_softmax_xent_scaled", dict(sim=None), (EINVAL, XENT)),
    ("n2_odd", "idl_nce_softmax_xent_scaled", dict(n2=3), (EINVAL, XENT)),
    ("temperature_nan", "idl_nce_softmax_xent_scaled", dict(temperature=NAN), (EINVAL, XENT)),

    ("valid", "idl_nce_normalize_backward", {}, (ECUDA, CUDA)),
    ("valid_wide", "idl_nce_normalize_backward", dict(D=200), (ECUDA, CUDA)),
    ("null_dfn", "idl_nce_normalize_backward", dict(dfn=None), (EINVAL, NBWD)),
    ("null_fn", "idl_nce_normalize_backward", dict(fn=None), (EINVAL, NBWD)),
    ("null_inv_norm", "idl_nce_normalize_backward", dict(inv_norm=None), (EINVAL, NBWD)),
    ("null_dh", "idl_nce_normalize_backward", dict(dh=None), (EINVAL, NBWD)),
    ("n2_0", "idl_nce_normalize_backward", dict(n2=0), (EINVAL, NBWD)),
    ("D_0", "idl_nce_normalize_backward", dict(D=0), (EINVAL, NBWD)),
    ("valid", "idl_nce_normalize_backward_parts", {}, (ECUDA, CUDA)),
    ("n_parts_0", "idl_nce_normalize_backward_parts", dict(n_parts=0), (EINVAL, NBWD)),
    ("null_dh", "idl_nce_normalize_backward_parts", dict(dh=None), (EINVAL, NBWD)),
    ("D_negative", "idl_nce_normalize_backward_parts", dict(D=-64), (EINVAL, NBWD)),

    ("valid", "idl_relu_dropout_forward", {}, (ECUDA, CUDA)),
    ("valid_no_bias_no_step", "idl_relu_dropout_forward", dict(bias=None, step=None, n_parts=1), (ECUDA, CUDA)),
    ("valid_p0", "idl_relu_dropout_forward", dict(p=0.0), (ECUDA, CUDA)),
    ("valid_p_below_1", "idl_relu_dropout_forward", dict(p=1.0 - 2.0 ** -24), (ECUDA, CUDA)),
    ("valid_N4_M1", "idl_relu_dropout_forward", dict(M=1, N=4), (ECUDA, CUDA)),
    ("valid_step_8_aligned", "idl_relu_dropout_forward", dict(step=DEV + 8), (ECUDA, CUDA)),
    ("null_parts", "idl_relu_dropout_forward", dict(parts=None), (EINVAL, FWD)),
    ("null_out", "idl_relu_dropout_forward", dict(out=None), (EINVAL, FWD)),
    ("n_parts_0", "idl_relu_dropout_forward", dict(n_parts=0), (EINVAL, FWD)),
    ("M_0", "idl_relu_dropout_forward", dict(M=0), (EINVAL, FWD)),
    ("N_0", "idl_relu_dropout_forward", dict(N=0), (EINVAL, FWD)),
    ("N_not_multiple_of_4", "idl_relu_dropout_forward", dict(N=514), (EINVAL, FWD)),
    ("p_1", "idl_relu_dropout_forward", dict(p=1.0), (EINVAL, FWD)),
    ("p_negative", "idl_relu_dropout_forward", dict(p=-0.1), (EINVAL, FWD)),
    ("p_nan", "idl_relu_dropout_forward", dict(p=NAN), (EINVAL, FWD)),
    ("misaligned_parts", "idl_relu_dropout_forward", dict(parts=ODD), (EINVAL, FWD_ALIGN)),
    ("misaligned_parts_8", "idl_relu_dropout_forward", dict(parts=DEV + 8), (EINVAL, FWD_ALIGN)),
    ("misaligned_bias", "idl_relu_dropout_forward", dict(bias=ODD), (EINVAL, FWD_ALIGN)),
    ("misaligned_out", "idl_relu_dropout_forward", dict(out=ODD), (EINVAL, FWD_ALIGN)),

    ("valid", "idl_relu_dropout_backward", {}, (ECUDA, CUDA)),
    ("valid_n4", "idl_relu_dropout_backward", dict(n=4), (ECUDA, CUDA)),
    ("null_out", "idl_relu_dropout_backward", dict(out=None), (EINVAL, BWD)),
    ("null_dy", "idl_relu_dropout_backward", dict(dy=None), (EINVAL, BWD)),
    ("null_dx", "idl_relu_dropout_backward", dict(dx=None), (EINVAL, BWD)),
    ("n_0", "idl_relu_dropout_backward", dict(n=0), (EINVAL, BWD)),
    ("n_not_multiple_of_4", "idl_relu_dropout_backward", dict(n=4098), (EINVAL, BWD)),
    ("p_1", "idl_relu_dropout_backward", dict(p=1.0), (EINVAL, BWD)),
    ("p_nan", "idl_relu_dropout_backward", dict(p=NAN), (EINVAL, BWD)),
    ("misaligned_out", "idl_relu_dropout_backward", dict(out=ODD), (EINVAL, BWD_ALIGN)),
    ("misaligned_dy", "idl_relu_dropout_backward", dict(dy=ODD), (EINVAL, BWD_ALIGN)),
    ("misaligned_dx", "idl_relu_dropout_backward", dict(dx=DEV + 8), (EINVAL, BWD_ALIGN)),

    ("valid", "idl_sum_parts_bias", {}, (ECUDA, CUDA)),
    ("valid_no_bias", "idl_sum_parts_bias", dict(bias=None), (ECUDA, CUDA)),
    ("null_parts", "idl_sum_parts_bias", dict(parts=None), (EINVAL, SUM)),
    ("null_out", "idl_sum_parts_bias", dict(out=None), (EINVAL, SUM)),
    ("n_parts_0", "idl_sum_parts_bias", dict(n_parts=0), (EINVAL, SUM)),
    ("M_0", "idl_sum_parts_bias", dict(M=0), (EINVAL, SUM)),
    ("N_2", "idl_sum_parts_bias", dict(N=2), (EINVAL, SUM)),
    ("N_not_multiple_of_4", "idl_sum_parts_bias", dict(N=66), (EINVAL, SUM)),
    ("misaligned_parts", "idl_sum_parts_bias", dict(parts=ODD), (EINVAL, SUM_ALIGN)),
    ("misaligned_bias", "idl_sum_parts_bias", dict(bias=DEV + 8), (EINVAL, SUM_ALIGN)),
    ("misaligned_out", "idl_sum_parts_bias", dict(out=ODD), (EINVAL, SUM_ALIGN)),

    ("valid", "idl_pair_selection", {}, (ECUDA, CUDA)),
    ("n_0", "idl_pair_selection", dict(n_pairs=0), (OK, None)),
    ("null_pair_ids", "idl_pair_selection", dict(pair_ids=None), (EINVAL, PAIR)),
    ("null_sidx", "idl_pair_selection", dict(sidx=None), (EINVAL, PAIR)),
    ("null_sel", "idl_pair_selection", dict(sel=None), (EINVAL, PAIR)),
    ("n_negative", "idl_pair_selection", dict(n_pairs=-1), (EINVAL, PAIR)),
    ("n_seqs_0", "idl_pair_selection", dict(n_seqs=0), (EINVAL, PAIR)),
    ("null_checked_when_n_0", "idl_pair_selection", dict(n_pairs=0, sel=None), (EINVAL, PAIR)),

    ("valid", "idl_rmsprop_step", {}, (ECUDA, CUDA)),
    ("valid_unaligned", "idl_rmsprop_step", dict(param=ODD, grad=ODD, sq=ODD, n=5), (ECUDA, CUDA)),
    ("n_0", "idl_rmsprop_step", dict(n=0), (OK, None)),
    ("null_param", "idl_rmsprop_step", dict(param=None), (EINVAL, RMS)),
    ("null_grad", "idl_rmsprop_step", dict(grad=None), (EINVAL, RMS)),
    ("null_sq", "idl_rmsprop_step", dict(sq=None), (EINVAL, RMS)),
    ("n_negative", "idl_rmsprop_step", dict(n=-1), (EINVAL, RMS)),

    ("valid", "idl_rmsprop_allreduce_step", {}, (ECUDA, CUDA)),
    ("valid_world_1", "idl_rmsprop_allreduce_step", dict(world=1, n_total=4), (ECUDA, CUDA)),
    ("valid_world_16_last_rank", "idl_rmsprop_allreduce_step", dict(world=16, rank=15, n_total=64), (ECUDA, CUDA)),
    ("valid_multicast", "idl_rmsprop_allreduce_step", dict(grad_mc=1 << 40, param_mc=(1 << 40) + 4096), (ECUDA, CUDA)),
    ("world_17", "idl_rmsprop_allreduce_step", dict(world=17, n_total=17 * 64), (EINVAL, AR)),
    ("world_0", "idl_rmsprop_allreduce_step", dict(world=0), (EINVAL, AR)),
    ("rank_negative", "idl_rmsprop_allreduce_step", dict(rank=-1), (EINVAL, AR)),
    ("rank_equals_world", "idl_rmsprop_allreduce_step", dict(rank=2), (EINVAL, AR)),
    ("n_total_0", "idl_rmsprop_allreduce_step", dict(n_total=0), (EINVAL, AR)),
    ("n_total_negative", "idl_rmsprop_allreduce_step", dict(n_total=-8), (EINVAL, AR)),
    ("n_total_not_multiple_of_4_world", "idl_rmsprop_allreduce_step", dict(n_total=1028), (EINVAL, AR)),
    ("n_total_3_world", "idl_rmsprop_allreduce_step", dict(world=3, n_total=3 * 4 * 5 + 4), (EINVAL, AR)),
    ("null_grad_table", "idl_rmsprop_allreduce_step", dict(grad_peers=None), (EINVAL, AR)),
    ("null_param_table", "idl_rmsprop_allreduce_step", dict(param_peers=None), (EINVAL, AR)),
    ("null_sq", "idl_rmsprop_allreduce_step", dict(sq=None), (EINVAL, AR)),
    ("null_grad_peer", "idl_rmsprop_allreduce_step", dict(grad_peers=dict(r1=0)), (EINVAL, AR_PEER)),
    ("null_param_peer", "idl_rmsprop_allreduce_step", dict(param_peers=dict(r0=0)), (EINVAL, AR_PEER)),
    ("misaligned_grad_peer", "idl_rmsprop_allreduce_step", dict(grad_peers=dict(r1=ODD)), (EINVAL, AR_PEER)),
    ("misaligned_param_peer", "idl_rmsprop_allreduce_step", dict(param_peers=dict(r0=DEV + 8)), (EINVAL, AR_PEER)),
    ("misaligned_sq", "idl_rmsprop_allreduce_step", dict(sq=ODD), (EINVAL, AR_ALIGN)),
    ("misaligned_sq_8", "idl_rmsprop_allreduce_step", dict(sq=DEV + 8), (EINVAL, AR_ALIGN)),
    ("misaligned_grad_multicast", "idl_rmsprop_allreduce_step", dict(grad_mc=(1 << 40) + 4, param_mc=1 << 40), (EINVAL, AR_ALIGN)),
    ("misaligned_param_multicast", "idl_rmsprop_allreduce_step", dict(grad_mc=1 << 40, param_mc=(1 << 40) + 8), (EINVAL, AR_ALIGN)),
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
def test_train_ops_entry_point_validation(called, case):
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
