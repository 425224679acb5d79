"""Quick kernel timing sweeps (CUDA events) for tuning; not the bench.  Usage on the GPU box:
   python tools/perf_probe.py scl|scl3|sptest|fe [n] [B]        (SC decoder: tools/sc_check.py)"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "polar-code-pytorch-sionna_b200")
for p in (ROOT, PKG, os.path.join(PKG, "x_run_sn_polar")):
    sys.path.insert(0, p)
import numpy as np
import torch

import d_kernels as dk
from oracle import polar_oracle as po


def timeit(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), float(np.median(ts))


def main():
    what = sys.argv[1] if len(sys.argv) > 1 else "scl3"
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
    k = n // 2
    dev = torch.device("cuda", 0)
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    no = po.ebnodb2no(4.0, 2, k / n)
    if what == "scl":
        L = int(os.environ.get("L", "8"))
        B = int(sys.argv[3]) if len(sys.argv) > 3 else 1 << 15
        _, _, x = dk.awgn_frontend(tables, B, no, 1234)
        best, med = timeit(lambda: dk.scl_decode(x, tables, L, want_packed=True, want_info=False), iters=3, warm=1)
        print("SCL L=%d n=%d B=%d: %8.3f ms  %.3e cw/s  %.3f Gbit/s info" %
              (L, n, B, best, B / best * 1e3, B / best * 1e3 * k / 1e9), flush=True)
    elif what == "sptest":
        import ctypes
        cnt = torch.zeros(3, dtype=torch.int64, device=dev)
        N = int(sys.argv[3]) if len(sys.argv) > 3 else 1 << 28
        dk.check(dk.lib().polar_scl3_math_selftest(N, dk.ptr(cnt), dk.stream_ptr(dev)))
        torch.cuda.synchronize()
        print("softplus selftest: %d arguments, mismatches exp/log/softplus vs CUDA math library:" % N, cnt.tolist(), flush=True)
    elif what == "scl3":
        # scl3 tuning sweep + differential check against scl2 on the same inputs (decisions, all PMs, lists)
        L = int(os.environ.get("L", "8"))
        B = int(sys.argv[3]) if len(sys.argv) > 3 else 1 << 15
        ebno = float(os.environ.get("EBNO", "3.0"))
        _, _, x = dk.awgn_frontend(tables, B, po.ebnodb2no(ebno, 2, k / n), 1234)
        dk.set_option("POLAR_SCL_MODE", int("1"))
        ref = dk.scl_decode(x, tables, L, want_packed=True, want_info=False, want_pm=True, want_list=True)
        torch.cuda.synchronize()
        best, med = timeit(lambda: dk.scl_decode(x, tables, L, want_packed=True, want_info=False), iters=3, warm=1)
        print("scl2 L=%d n=%d B=%d: %8.3f ms  %.3e cw/s  %.3f Gbit/s info" % (L, n, B, best, B / best * 1e3, B / best * 1e3 * k / 1e9), flush=True)
        dk.set_option("POLAR_SCL_MODE", int("2"))
        for ss in [int(v) for v in os.environ.get("SS", "5,6,7").split(",")]:
            for ctas in [int(v) for v in os.environ.get("CTAS", "0").split(",")]:
                dk.set_option("POLAR_SCL3_SS", int(str(ss))); dk.set_option("POLAR_SCL3_CTAS", int(str(ctas)))
                try:
                    got = dk.scl_decode(x, tables, L, want_packed=True, want_info=False, want_pm=True, want_list=True)
                    torch.cuda.synchronize()
                    d_best = int((got["u_packed"] != ref["u_packed"]).any(dim=1).sum())
                    d_list = int((got["list"] != ref["list"]).any(dim=2).any(dim=1).sum())
                    rel = ((got["pm"] - ref["pm"]).abs() / ref["pm"].abs().clamp_min(1e-30)).max().item()
                    best, med = timeit(lambda: dk.scl_decode(x, tables, L, want_packed=True, want_info=False), iters=3, warm=1)
                    print("scl3 L=%d n=%d B=%d SS=%d ctas=%d: %8.3f ms  %.3e cw/s  %.3f Gbit/s info | vs scl2: best-path diffs %d, list diffs %d, max rel pm %.2e" %
                          (L, n, B, ss, ctas, best, B / best * 1e3, B / best * 1e3 * k / 1e9, d_best, d_list, rel), flush=True)
                except Exception as e:
                    print("scl3 SS=%d ctas=%d failed: %s" % (ss, ctas, e), flush=True)
    elif what == "fe":
        B = int(sys.argv[3]) if len(sys.argv) > 3 else (1 << 28) // n
        f = lambda: dk.awgn_frontend(tables, B, no, 1234)
        best, med = timeit(f)
        print("frontend n=%d B=%d: %.3f ms  %.3e cw/s  write %.1f GB/s" % (n, B, best, B / best * 1e3, B * n * 4 / best * 1e3 / 1e9))


if __name__ == "__main__":
    main()
