"""Argument validation of the global-batch loss entry points of the C ABI (idl_iid_partial_s2, idl_iid_global_finish,
idl_nce_gather_rows, idl_nce_softmax_xent_rows, idl_nce_normalize_backward_global): the return code and the exact idl_last_error()
text of every argument set below.

As in test_train_ops_abi_validation.py the calls run in a child process with CUDA_VISIBLE_DEVICES="", so a request that passes
validation fails at its first CUDA call with IDL_ECUDA instead of launching on the placeholder pointers: a missing check shows up
as a CUDA error here, never as a fault.  The kernels read the peers' buffers as floats, so a peer address must be non-null and
4-byte aligned; the row counts must keep the [2B, D] and [2b, 2B] operands indexable with 32-bit rows."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OK, EINVAL, ECUDA = 0, 1, 2
DEV = 64    # placeholder device pointer (16-byte aligned)
ORDER = {
    "idl_iid_partial_s2": "z1 z2 B C S2 stream",
    "idl_iid_global_finish": "peers world z1 z2 B C lamb eps grad_scale loss_weight add add_weight loss dz1 dz2 ws ws_bytes stream",
    "idl_nce_gather_rows": "peers world b D fn_all stream",
    "idl_nce_softmax_xent_rows": "sim b rank world temperature grad_scale rowloss stream",
    "idl_nce_normalize_backward_global": "dfn n_parts peers world fn inv_norm b D rank dh loss stream",
}
BASE = dict(z1=DEV, z2=DEV, B=64, C=5, S2=DEV, peers="world", world=2, lamb=2.8, eps=2.2e-16, grad_scale=0.5, loss_weight=0.25, add=DEV,
            add_weight=0.75, loss=DEV, dz1=DEV, dz2=DEV, ws=DEV, ws_bytes=1 << 20, b=64, D=64, fn_all=DEV, sim=DEV, rank=1, temperature=0.85,
            rowloss=DEV, dfn=DEV, n_parts=1, fn=DEV, inv_norm=DEV, dh=DEV, stream=None)
POINTERS = set("z1 z2 S2 add loss dz1 dz2 ws fn_all sim rowloss dfn fn inv_norm dh stream".split())
CUDA = "<cuda>"   # any CUDA runtime error: the request got past validation

PS2 = "idl_iid_partial_s2: bad argument (B >= 1, 1 <= C <= 256)"
FIN = "idl_iid_global_finish: bad argument (world 1..16, B >= 1, 1 <= C <= 256)"
FIN_WS = "idl_iid_global_finish: workspace too small"
FIN_PEER = "idl_iid_global_finish: null / misaligned peer pointer"
GAT = "idl_nce_gather_rows: bad argument (world 1..16, b >= 1, D >= 1, 2 b world D < 2^31)"
GAT_PEER = "idl_nce_gather_rows: null / misaligned peer pointer"
ROWS = "idl_nce_softmax_xent_rows: bad argument (world 1..16, 0 <= rank < world, b >= 1, 4 b^2 world^2 < 2^31)"
GBWD = "idl_nce_normalize_backward_global: bad argument (world 1..16, 0 <= rank < world, b >= 1, 1 <= D <= 128)"
GBWD_PEER = "idl_nce_normalize_backward_global: null / misaligned peer pointer"


def _peers(world, **at):
    """placeholder peer table of `world` ranks (distinct aligned addresses); at = {rank: address} overrides"""
    return [at.get("r%d" % r, DEV * (r + 1)) for r in range(world)]


# (id, entry point, arguments that differ from BASE, (return code, error text or CUDA or None))
CASES = [
    ("valid", "idl_iid_partial_s2", {}, (ECUDA, CUDA)),
    ("valid_C_1", "idl_iid_partial_s2", dict(C=1), (ECUDA, CUDA)),
    ("valid_C_256", "idl_iid_partial_s2", dict(C=256), (ECUDA, CUDA)),
    ("valid_B_1", "idl_iid_partial_s2", dict(B=1), (ECUDA, CUDA)),
    ("null_z1", "idl_iid_partial_s2", dict(z1=None), (EINVAL, PS2)),
    ("null_z2", "idl_iid_partial_s2", dict(z2=None), (EINVAL, PS2)),
    ("null_S2", "idl_iid_partial_s2", dict(S2=None), (EINVAL, PS2)),
    ("B_0", "idl_iid_partial_s2", dict(B=0), (EINVAL, PS2)),
    ("C_0", "idl_iid_partial_s2", dict(C=0), (EINVAL, PS2)),
    ("C_257", "idl_iid_partial_s2", dict(C=257), (EINVAL, PS2)),

    ("valid", "idl_iid_global_finish", {}, (ECUDA, CUDA)),
    ("valid_C_16", "idl_iid_global_finish", dict(C=16), (ECUDA, CUDA)),
    ("valid_C_17", "idl_iid_global_finish", dict(C=17), (ECUDA, CUDA)),
    ("valid_C_256", "idl_iid_global_finish", dict(C=256), (ECUDA, CUDA)),
    ("valid_world_1", "idl_iid_global_finish", dict(world=1), (ECUDA, CUDA)),
    ("valid_world_16", "idl_iid_global_finish", dict(world=16), (ECUDA, CUDA)),
    ("valid_no_outputs", "idl_iid_global_finish", dict(add=None, loss=None, dz1=None, dz2=None), (ECUDA, CUDA)),
    ("valid_peer_4_aligned", "idl_iid_global_finish", dict(peers=dict(r1=DEV + 4)), (ECUDA, CUDA)),
    ("valid_exact_workspace_C_5", "idl_iid_global_finish", dict(ws_bytes=4 * (3 + 512 + 25) + 64), (ECUDA, CUDA)),
    ("valid_exact_workspace_C_200", "idl_iid_global_finish", dict(C=200, ws_bytes=4 * (2 * 200 * 200 + 6 * 200)), (ECUDA, CUDA)),
    ("workspace_short_C_5", "idl_iid_global_finish", dict(ws_bytes=4 * (3 + 512 + 25) + 63), (EINVAL, FIN_WS)),
    ("workspace_short_C_200", "idl_iid_global_finish", dict(C=200, ws_bytes=4 * (2 * 200 * 200 + 6 * 200) - 1), (EINVAL, FIN_WS)),
    ("null_table", "idl_iid_global_finish", dict(peers=None), (EINVAL, FIN)),
    ("null_z1", "idl_iid_global_finish", dict(z1=None), (EINVAL, FIN)),
    ("null_z2", "idl_iid_global_finish", dict(z2=None), (EINVAL, FIN)),
    ("null_workspace", "idl_iid_global_finish", dict(ws=None), (EINVAL, FIN)),
    ("world_0", "idl_iid_global_finish", dict(world=0), (EINVAL, FIN)),
    ("world_17", "idl_iid_global_finish", dict(world=17), (EINVAL, FIN)),
    ("B_0", "idl_iid_global_finish", dict(B=0), (EINVAL, FIN)),
    ("C_0", "idl_iid_global_finish", dict(C=0), (EINVAL, FIN)),
    ("C_257", "idl_iid_global_finish", dict(C=257), (EINVAL, FIN)),
    ("null_peer", "idl_iid_global_finish", dict(peers=dict(r1=0)), (EINVAL, FIN_PEER)),
    ("misaligned_peer", "idl_iid_global_finish", dict(peers=dict(r0=DEV + 2)), (EINVAL, FIN_PEER)),

    ("valid", "idl_nce_gather_rows", {}, (ECUDA, CUDA)),
    ("valid_world_16_odd_rows", "idl_nce_gather_rows", dict(world=16, b=37, D=3), (ECUDA, CUDA)),
    ("valid_largest", "idl_nce_gather_rows", dict(world=2, b=2 ** 23 - 1, D=64), (ECUDA, CUDA)),
    ("rows_overflow", "idl_nce_gather_rows", dict(world=2, b=2 ** 23, D=64), (EINVAL, GAT)),
    ("null_table", "idl_nce_gather_rows", dict(peers=None), (EINVAL, GAT)),
    ("null_out", "idl_nce_gather_rows", dict(fn_all=None), (EINVAL, GAT)),
    ("world_0", "idl_nce_gather_rows", dict(world=0), (EINVAL, GAT)),
    ("world_17", "idl_nce_gather_rows", dict(world=17), (EINVAL, GAT)),
    ("b_0", "idl_nce_gather_rows", dict(b=0), (EINVAL, GAT)),
    ("D_0", "idl_nce_gather_rows", dict(D=0), (EINVAL, GAT)),
    ("null_peer", "idl_nce_gather_rows", dict(peers=dict(r0=0)), (EINVAL, GAT_PEER)),
    ("misaligned_peer", "idl_nce_gather_rows", dict(peers=dict(r1=DEV + 1)), (EINVAL, GAT_PEER)),

    ("valid", "idl_nce_softmax_xent_rows", {}, (ECUDA, CUDA)),
    ("valid_rank_0", "idl_nce_softmax_xent_rows", dict(rank=0), (ECUDA, CUDA)),
    ("valid_world_1", "idl_nce_softmax_xent_rows", dict(world=1, rank=0, b=1), (ECUDA, CUDA)),
    ("valid_8_ranks_of_512", "idl_nce_softmax_xent_rows", dict(world=8, rank=7, b=512), (ECUDA, CUDA)),
    ("valid_largest", "idl_nce_softmax_xent_rows", dict(world=1, rank=0, b=23170), (ECUDA, CUDA)),
    ("rows_overflow", "idl_nce_softmax_xent_rows", dict(world=1, rank=0, b=23171), (EINVAL, ROWS)),
    ("null_sim", "idl_nce_softmax_xent_rows", dict(sim=None), (EINVAL, ROWS)),
    ("null_rowloss", "idl_nce_softmax_xent_rows", dict(rowloss=None), (EINVAL, ROWS)),
    ("temperature_0", "idl_nce_softmax_xent_rows", dict(temperature=0.0), (EINVAL, ROWS)),
    ("temperature_nan", "idl_nce_softmax_xent_rows", dict(temperature=float("nan")), (EINVAL, ROWS)),
    ("rank_negative", "idl_nce_softmax_xent_rows", dict(rank=-1), (EINVAL, ROWS)),
    ("rank_equals_world", "idl_nce_softmax_xent_rows", dict(rank=2), (EINVAL, ROWS)),
    ("world_0", "idl_nce_softmax_xent_rows", dict(world=0, rank=0), (EINVAL, ROWS)),
    ("world_17", "idl_nce_softmax_xent_rows", dict(world=17), (EINVAL, ROWS)),
    ("b_0", "idl_nce_softmax_xent_rows", dict(b=0), (EINVAL, ROWS)),

    ("valid", "idl_nce_normalize_backward_global", {}, (ECUDA, CUDA)),
    ("valid_no_loss", "idl_nce_normalize_backward_global", dict(loss=None), (ECUDA, CUDA)),
    ("valid_D_128_parts_8", "idl_nce_normalize_backward_global", dict(D=128, n_parts=8), (ECUDA, CUDA)),
    ("valid_world_16", "idl_nce_normalize_backward_global", dict(world=16, rank=15), (ECUDA, CUDA)),
    ("D_129", "idl_nce_normalize_backward_global", dict(D=129), (EINVAL, GBWD)),
    ("D_0", "idl_nce_normalize_backward_global", dict(D=0), (EINVAL, GBWD)),
    ("n_parts_0", "idl_nce_normalize_backward_global", dict(n_parts=0), (EINVAL, GBWD)),
    ("null_dfn", "idl_nce_normalize_backward_global", dict(dfn=None), (EINVAL, GBWD)),
    ("null_table", "idl_nce_normalize_backward_global", dict(peers=None), (EINVAL, GBWD)),
    ("null_fn", "idl_nce_normalize_backward_global", dict(fn=None), (EINVAL, GBWD)),
    ("null_inv_norm", "idl_nce_normalize_backward_global", dict(inv_norm=None), (EINVAL, GBWD)),
    ("null_dh", "idl_nce_normalize_backward_global", dict(dh=None), (EINVAL, GBWD)),
    ("rank_negative", "idl_nce_normalize_backward_global", dict(rank=-1), (EINVAL, GBWD)),
    ("rank_equals_world", "idl_nce_normalize_backward_global", dict(rank=2), (EINVAL, GBWD)),
    ("world_17", "idl_nce_normalize_backward_global", dict(world=17), (EINVAL, GBWD)),
    ("b_0", "idl_nce_normalize_backward_global", dict(b=0), (EINVAL, GBWD)),
    ("rows_overflow", "idl_nce_normalize_backward_global", dict(world=16, rank=0, b=2 ** 20, D=64), (EINVAL, GBWD)),
    ("null_peer", "idl_nce_normalize_backward_global", dict(peers=dict(r1=0)), (EINVAL, GBWD_PEER)),
    ("misaligned_peer", "idl_nce_normalize_backward_global", dict(peers=dict(r0=DEV + 6)), (EINVAL, GBWD_PEER)),
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
            if name == "peers" and v is not None:
                table = _peers(max(a["world"], 1), **(v if isinstance(v, dict) else {}))
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
def test_global_loss_entry_point_validation(called, case):
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
