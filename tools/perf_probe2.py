"""Timing of the whole-schedule featurisation kernel only (development aid)."""
import sys, os
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from idelucs_b200 import featurise as ft
from idelucs_b200.seqset import SeqSet

def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
    L = int(sys.argv[2]) if len(sys.argv) > 2 else 10000
    n_mimics = int(sys.argv[3]) if len(sys.argv) > 3 else 50
    k, F = 6, 4096
    g = torch.Generator(device="cuda").manual_seed(0)
    codes = torch.randint(0, 4, (n * L,), device="cuda", dtype=torch.uint8, generator=g)
    ascii_t = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")[codes.long()]
    del codes
    ss = SeqSet.from_ascii(ascii_t, np.arange(n + 1, dtype=np.int64) * L)
    variants = ft.mimic_schedule(n_mimics)
    V = len(variants)
    out = torch.empty((V, n, F), dtype=torch.float32, device="cuda")
    off = [v * n * F for v in range(V)]
    stride = F
    if os.environ.get("ITEM_MAJOR"):   # [N, V, F] instead of [V, N, F]
        off = [v * F for v in range(V)]
        stride = V * F
    mean = torch.rand(F, device="cuda") * 1e-3
    scale = torch.rand(F, device="cuda") * 1e-4 + 1e-5
    for name, kind, vs in (("48 random_n std", ft.OUT_STD_F32, variants[3:]), ("all %d std" % V, ft.OUT_STD_F32, variants)):
        nv = len(vs)
        prep = ft.prepare(ss, k, vs, seed=1) if ft.can_prepare(ss, k, vs) else None   # the k = 6 fast path reads the prepared deltas
        fn = lambda: ft.profiles(ss, k, vs, out_kind=kind, seed=1, out=out, out_off=off[:nv], out_stride=stride, mean=mean, scale=scale, prepared=prep)
        fn(); torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        by = nv * n * F * 4 + n * L / 4
        print("%-20s best %.3f ms  %.1f GB/s" % (name, min(ts), by / min(ts) / 1e6))
        if name.startswith("all"):
            fs = lambda: ft.prepare(ss, k, variants, seed=1)
            fs(); torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fs(); b.record(); torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            print("%-20s best %.3f ms" % ("prepare pass", min(ts)))
main()
