"""Hybrid SC -> SCL (polar_scl_decode_hybrid) against the full CRC-aided list decoder of the same arithmetic, configs[2] code
(k = 512 incl. CRC11, n = 1024, L = 8), B = 2^18 codewords with a valid CRC through the device QPSK/AWGN channel.

For each Eb/N0 and arithmetic (cn_mode 0: min-sum, full path polar_scl_decode -> scl3; cn_mode 2: boxplus with fast-SCL
pruning, full path polar_scl_decode_boxplus_pruned): list-decoded fraction, codewords/s of the hybrid and of the full
decode (CUDA events, the two alternating after warm-up, median of REPS each), codewords/s of the SC stage alone, and the
BLER of both.  Writes a markdown table.

  python tools/hybrid_probe.py [--out profiles/r03_hybrid.md] [--reps 5]"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "polar-code-pytorch-sionna_b200")
for p in (ROOT, PKG, os.path.join(PKG, "x_run_sn_polar")):
    sys.path.insert(0, p)
import numpy as np
import torch
import d_kernels as dk
from my_sn.fec.crc import CRCEncoder
from oracle import polar_oracle as po

N, K, L, CRC, B = 1024, 512, 8, "CRC11", 1 << 18
# the configs[2] code is the Reed-Muller-ranked one of bench.py, weak under SC: its list-decoded fraction reaches 1 % only
# above 4 dB, so the sweep continues to 8 dB
EBNOS = (0.0, 1.0, 1.5, 2.0, 2.5, 3.0, 4.0, 5.0, 6.0, 7.0, 8.0)
MODES = {0: "min-sum", 2: "boxplus pruned"}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_hybrid.md"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "hybrid_probe needs a CUDA device"
    dev = torch.device("cuda", 0)
    gpu = card()
    print("card:", gpu, flush=True)
    tables = dk.code_tables(po.rm_frozen_pos(N, N - K), N, dev)
    chk = CRCEncoder(CRC, K)
    gen = CRCEncoder(CRC, K - chk.crc_length)
    rows = torch.from_numpy(chk.syndrome_rows(tables.info_pos_np, N).view(np.int32).copy()).to(dev)
    nw = dk.words(N)
    out_h = torch.empty((B, nw), dtype=torch.int32, device=dev)
    out_f = torch.empty((B, nw), dtype=torch.int32, device=dev)
    out_s = torch.empty((B, nw), dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    res = []
    for ebno in EBNOS:
        torch.manual_seed(int(ebno * 10) + 1)
        bits = gen(torch.randint(0, 2, (B, K - gen.crc_length), device=dev, dtype=torch.float32))
        lg = dk.qpsk_awgn_llr(dk.encode_f32(bits, tables), po.ebnodb2no(ebno, 2, K / N), 1234 + int(ebno * 10))
        full_tx = torch.zeros((B, N), dtype=torch.float32, device=dev)
        full_tx[:, tables.info_pos.long()] = bits
        tx = dk.pack_bits(full_tx)
        del full_tx, bits

        def bler(hat):
            c = torch.zeros(2, dtype=torch.int64, device=dev)
            dk.count_errors_packed(tx, hat, tables.info_mask, N, c)
            return c[1].item() / B

        for mode, name in MODES.items():
            box = mode != 0
            hyb = lambda: dk.scl_decode_hybrid(lg, tables, L, rows, chk.crc_length, mode, want_info=False, out_packed=out_h,
                                               n_list_out=cnt)
            full = lambda: dk.scl_decode(lg, tables, L, crc_rows=rows, crc_len=chk.crc_length, want_info=False,
                                         out_packed=out_f, boxplus=box, pruned=box)
            sc = lambda: dk.sc_decode(lg, tables, want_info=False, out_packed=out_s, boxplus=box)
            for f in (hyb, full, sc, hyb, full):
                f()
            torch.cuda.synchronize()
            th, tf, ts = [], [], []
            for _ in range(args.reps):
                th.append(timed(hyb)); tf.append(timed(full)); ts.append(timed(sc))
            r = dict(ebno=ebno, mode=name, rows=cnt.item(), frac=cnt.item() / B, hyb_ms=float(np.median(th)), full_ms=float(np.median(tf)),
                     sc_ms=float(np.median(ts)), bler_h=bler(out_h), bler_f=bler(out_f))
            r["speedup"] = r["full_ms"] / r["hyb_ms"]
            res.append(r)
            print("Eb/N0 %.1f dB %-14s list-decoded %.3e  hybrid %.2f ms (%.3e cw/s)  full %.2f ms (%.3e cw/s)  x%.2f  "
                  "SC %.2f ms  BLER hybrid %.3e full %.3e" % (ebno, name, r["frac"], r["hyb_ms"], B / r["hyb_ms"] * 1e3,
                                                              r["full_ms"], B / r["full_ms"] * 1e3, r["speedup"], r["sc_ms"],
                                                              r["bler_h"], r["bler_f"]), flush=True)
        del lg, tx
    lines = ["# Hybrid SC -> SCL vs full CRC-aided SCL, configs[2] code (k = 512 incl. CRC11, n = 1024, L = 8), B = 2^18",
             "",
             "Measured with `python tools/hybrid_probe.py` on: %s (name, power limit, max SM clock)." % gpu,
             "Codewords carry a valid CRC11 and go through the device QPSK/AWGN channel; each Eb/N0 has its own seeded batch.",
             "Times are CUDA-event medians of %d decodes of the whole batch, hybrid and full decode alternating after warm-up;"
             " SC is the SC stage alone (the same kernel the hybrid starts with).  Full decode: min-sum = `polar_scl_decode`"
             " (scl3), boxplus pruned = `polar_scl_decode_boxplus_pruned` (scl2 with fast-SCL pruning).  The hybrid's list"
             " stage is scl2 in both arithmetics." % args.reps,
             "",
             "| Eb/N0 (dB) | arithmetic | list-decoded rows | fraction | hybrid ms | hybrid cw/s | full ms | full cw/s |"
             " speed-up | SC ms | hybrid - SC ms | BLER hybrid | BLER full |",
             "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in res:
        lines.append("| %.1f | %s | %d | %.2e | %.2f | %.3e | %.2f | %.3e | %.2fx | %.2f | %.2f | %.3e | %.3e |" % (
            r["ebno"], r["mode"], r["rows"], r["frac"], r["hyb_ms"], B / r["hyb_ms"] * 1e3, r["full_ms"], B / r["full_ms"] * 1e3,
            r["speedup"], r["sc_ms"], r["hyb_ms"] - r["sc_ms"], r["bler_h"], r["bler_f"]))
    lines.append("")
    for name in MODES.values():
        low = [r for r in res if r["mode"] == name and r["frac"] <= 0.01]
        if low:
            r = min(low, key=lambda r: r["ebno"])
            lines.append("%s: lowest Eb/N0 with a list-decoded fraction <= 1 %% is %.1f dB (%.2e): hybrid %.2fx the full "
                         "decode; hybrid - SC = %.2f ms for the CRC check and the list stage." % (
                             name, r["ebno"], r["frac"], r["speedup"], r["hyb_ms"] - r["sc_ms"]))
        else:
            lines.append("%s: no Eb/N0 point with a list-decoded fraction <= 1 %%." % name)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines[-len(MODES):]))
    print("wrote", args.out)


if __name__ == "__main__":
    main()
