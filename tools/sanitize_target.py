"""Small invocation of every hand-written kernel family, for compute-sanitizer (racecheck / synccheck / memcheck):
prepare pass + producer/consumer kernel (TMA bulk copies, mbarriers), generic kernel (short + int32 long path), chunked
long-genome path, IIC loss (single-CTA kernels, GEMM route, the C ABI's contraction kernels), fused InfoNCE, RMSprop.  Results are compared with the generic
kernel so that a sanitizer-clean run is also a correct one."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from idelucs_b200 import featurise as ft
from idelucs_b200.LossFunctions import IID_loss, info_nce_loss
from idelucs_b200.seqset import SeqSet


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    rng = np.random.default_rng(0)
    alph = np.frombuffer(b"ACGTACGTACGTACGTN", dtype=np.uint8)
    if which in ("all", "schedule"):
        seqs = [alph[rng.integers(0, alph.size, size=int(L))].tobytes() for L in rng.integers(200, 1500, size=320)]
        ss = SeqSet.from_sequences(seqs)
        variants = ft.mimic_schedule(50)
        x, sc = ft.schedule_profiles(ss, 6, variants, out_kind=ft.OUT_STD_F32, seed=3)
        y, sc2 = ft.schedule_profiles(ss, 6, variants, out_kind=ft.OUT_STD_F32, seed=3, fast=False)
        torch.cuda.synchronize()
        assert torch.allclose(sc.mean64, sc2.mean64, rtol=1e-12)
        y2 = ft.profiles(ss, 6, variants, out_kind=ft.OUT_STD_F32, seed=3, mean=sc.mean32, scale=sc.scale32)
        assert torch.equal(x, y2)
        print("schedule ok", tuple(x.shape))
    if which in ("all", "long"):
        seqs = [alph[rng.integers(0, alph.size, size=int(L))].tobytes() for L in (70000, 3000, 140000, 66000)]
        ss = SeqSet.from_sequences(seqs)
        variants = ft.mimic_schedule(4)
        a = ft.profiles(ss, 6, variants, out_kind=ft.OUT_COUNTS_I32, seed=5)
        b = ft.profiles(ss, 6, variants, out_kind=ft.OUT_COUNTS_I32, seed=5, chunked=False)
        torch.cuda.synchronize()
        assert torch.equal(a, b)
        print("long ok")
    if which in ("all", "loss"):
        for B, C in ((96, 5), (700, 8), (96, 12), (96, 40)):   # register kernel (one / several rows per thread), single-CTA kernel, GEMM route
            z1 = torch.softmax(torch.randn(B, C, device="cuda"), 1).requires_grad_(True)
            z2 = torch.softmax(torch.randn(B, C, device="cuda"), 1).requires_grad_(True)
            IID_loss(z1, z2, lamb=2.8).backward()
        from idelucs_b200.LossFunctions import train_losses_and_grads
        for B, C in ((512, 5), (37, 3)):   # weighted path: vectorised / scalar weights kernel, split / single gradient GEMM
            z = torch.softmax(torch.randn(2 * B, C, device="cuda"), 1)
            h = torch.randn(2 * B, 64, device="cuda")
            train_losses_and_grads(z, h, 2.8, 0.25, 0.85)
        h1 = torch.randn(64, 64, device="cuda", requires_grad=True)
        h2 = torch.randn(64, 64, device="cuda", requires_grad=True)
        info_nce_loss(h1, h2, 0.85).backward()
        from idelucs_b200 import _lib
        lib = _lib.load()
        p, g, v = torch.randn(1000, device="cuda"), torch.randn(1000, device="cuda"), torch.zeros(1000, device="cuda")
        _lib.check(lib.idl_rmsprop_step(_lib.ptr(p), _lib.ptr(g), _lib.ptr(v), 1000, 1e-3, 0.99, 1e-8, 0.01, 1.0, _lib.stream_ptr()))
        # the C ABI's own contraction kernels around the algebra kernels (the Python layer takes the GEMM route above 16 clusters)
        from idelucs_b200.LossFunctions import _ws
        z1 = torch.softmax(torch.randn(96, 40, device="cuda"), 1); z2 = torch.softmax(torch.randn(96, 40, device="cuda"), 1)
        lo = torch.empty((), device="cuda"); d1 = torch.empty_like(z1); d2 = torch.empty_like(z2); ws = _ws(z1.device, 40)
        _lib.check(lib.idl_iid_loss(_lib.ptr(z1), _lib.ptr(z2), 96, 40, 2.8, 2.2e-16, _lib.ptr(lo), None, _lib.ptr(d1), _lib.ptr(d2), _lib.ptr(ws),
                                    ws.numel(), _lib.stream_ptr()))
        # two eager training steps: fused ReLU - Dropout kernels, pair selection, capped featurisation on the side stream, optimiser
        from idelucs_b200.train import ShardedTrainer
        seqs = [alph[rng.integers(0, 4, size=400)].tobytes() for _ in range(300)]
        tr = ShardedTrainer(SeqSet.from_sequences(seqs), k=6, n_clusters=5, n_mimics=3, batch_sz=64, seed=2)
        for _ in range(2):
            tr.step()
        ids = torch.randint(0, 5000, (300,), device="cuda")
        sidx = torch.empty(300, dtype=torch.int32, device="cuda"); sel = torch.empty((300, 2), dtype=torch.int32, device="cuda")
        _lib.check(lib.idl_pair_selection(_lib.ptr(ids), 300, 100, _lib.ptr(sidx), _lib.ptr(sel), _lib.stream_ptr()))
        torch.cuda.synchronize()
        assert torch.equal(sidx.long(), ids % 100) and torch.equal(sel[:, 1].long(), ids // 100 + 1)
        print("loss ok")


main()
