"""Quick device-side timing of the featurisation kernels (development aid, not the bench)."""
import sys
import time
import os

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from idelucs_b200 import featurise as ft
from idelucs_b200.seqset import SeqSet


def timeit(fn, iters=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), sum(ts) / len(ts)


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
    L = int(sys.argv[2]) if len(sys.argv) > 2 else 10000
    n_mimics = int(sys.argv[3]) if len(sys.argv) > 3 else 50
    k = int(sys.argv[4]) if len(sys.argv) > 4 else 6
    F = 4 ** k
    g = torch.Generator(device="cuda").manual_seed(0)
    codes = torch.randint(0, 4, (n * L,), device="cuda", dtype=torch.uint8, generator=g)
    ascii_t = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")[codes.long()]
    del codes
    t0 = time.time()
    ss = SeqSet.from_ascii(ascii_t, np.arange(n + 1, dtype=np.int64) * L)
    torch.cuda.synchronize()
    print("pack: %.1f ms (incl. alloc)" % ((time.time() - t0) * 1e3))
    variants = ft.mimic_schedule(n_mimics)
    V = len(variants)
    out = torch.empty((V, n, F), dtype=torch.float32, device="cuda")
    off = [v * n * F for v in range(V)]
    mean = torch.zeros(F, device="cuda")
    scale = torch.ones(F, device="cuda")
    bytes_out = V * n * F * 4
    for name, kind, vs in (("clean counts only", ft.OUT_COUNTS_I32, [ft.VariantSpec(ft.KIND_CLEAN)]),
                           ("t_norm freq (pass 0)", ft.OUT_FREQ_F32, variants[:1]),
                           ("3 bernoulli passes", ft.OUT_FREQ_F32, variants[:3]),
                           ("48 random_n passes", ft.OUT_FREQ_F32, variants[3:]),
                           ("all %d variants freq" % V, ft.OUT_FREQ_F32, variants),
                           ("all %d variants std" % V, ft.OUT_STD_F32, variants)):
        nv = len(vs)
        o = out.view(torch.int32) if kind == ft.OUT_COUNTS_I32 else out
        prep = None
        if kind != ft.OUT_COUNTS_I32 and ft.can_prepare(ss, k, vs):
            best, avg = timeit(lambda: ft.prepare(ss, k, vs, seed=1))
            print("%-28s best %8.3f ms avg %8.3f ms   (prepare pass incl. statistics)" % (name, best, avg))
            prep = ft.prepare(ss, k, vs, seed=1)
        best, avg = timeit(lambda: ft.profiles(ss, k, vs, out_kind=kind, seed=1, out=o, out_off=off[:nv], out_stride=F,
                                               mean=mean, scale=scale, prepared=prep))
        b = nv * n * F * 4 + n * L / 4
        print("%-28s best %8.3f ms avg %8.3f ms  %8.1f Mprofiles/s  %7.1f GB/s" % (name, best, avg, nv * n / best / 1e3, b / best / 1e6))
    best, avg = timeit(lambda: ft.Scaler.fit(out[0]))
    print("scaler fit on [%d,%d]: %.3f ms" % (n, F, best))
    big = out[:8]
    best, avg = timeit(lambda: big.fill_(1.0))
    print("torch fill 8 variants (write only): %.3f ms -> %.1f GB/s" % (best, big.numel() * 4 / best / 1e6))
    best, avg = timeit(lambda: big.sum())
    print("torch sum 8 variants (read only): %.3f ms -> %.1f GB/s" % (best, big.numel() * 4 / best / 1e6))
    best, avg = timeit(lambda: out[1].copy_(out[0]))
    print("torch copy 1 variant: %.3f ms -> %.1f GB/s" % (best, 2 * n * F * 4 / best / 1e6))


if __name__ == "__main__":
    main()
