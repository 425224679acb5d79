"""Belief-propagation decoder (`polar_belief_decode_f32`): kernel throughput against its shared-memory and issue bounds,
and device-loop BLER sweeps next to SC and SCL-8.

Throughput: (n, k) = (64, 32), (256, 128), (1024, 512), 5 and 20 iterations, min-sum and boxplus.  256 MB of logits per
launch (twice the 126 MB L2), CUDA-event median of REPS launches after warm-up, packed output only.  PE updates per
codeword as the kernel runs them: ((2T - 1)(m - 1) + 1) n/2 (the right-to-left stage 0 runs in the last iteration only,
the last left-to-right sweep is skipped); one PE update is two f evaluations.

Bounds, from the SM clock read in the same run (nvidia-smi clocks.max.sm) and 148 SMs:
  - shared memory: 24 B per PE update (four fp32 loads, two stores) at 128 B/clk/SM;
  - issue: the static SASS length of the kernel's two stage loops (cuobjdump -sass), one warp instruction per 32 PE
    updates per loop instruction, at 4 warp instructions/clk/SM;
  - MUFU (exp2 / log2, boxplus only): MUFU instructions of the same loops at 16 per clk/SM.

Sweeps: sim_ber on the device loop, target 1000 block errors, at most MAX_ITER iterations of BS codewords per point.

  python tools/bp_probe.py [--out profiles/r05_bp.md] [--reps 10]"""
import argparse
import os
import re
import subprocess
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
from my_sn.fec.polar.dec import BP_Dec, Polar5GDecoder
from my_sn.fec.polar.enc import Polar5GEncoder
from my_sn.sim import sim_ber
from my_sn.trans import ebno as ebno_mod
from polar.enc import PolarEncoder
from polar.polar_sc import SC_Dec
from polar.polar_scl import SCL_Dec
from z_sys_model.awgn_model import System_AWGN_model

CODES = ((64, 32), (256, 128), (1024, 512))
ITERS = (5, 20)
BYTES_IN = 1 << 28
SMS, SMEM_B_PER_CLK, ISSUE_PER_CLK, MUFU_PER_CLK = 148, 128, 4, 16
BS, MAX_ITER, TARGET = 1 << 14, 30, 1000


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return name, power, float(clk.split()[0]) * 1e6


def median_ms(fn, reps):
    fn(); fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def loop_sass(so):
    """{namespace: (instructions, MUFU instructions)} of the two stage loops of each belief_kernel build: the innermost
    loops (a backward branch with no other backward branch inside) whose body holds the stage barrier (BAR)."""
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    res = {}
    for fn in re.split(r"Function : ", out)[1:]:
        name = fn.split("\n", 1)[0]
        if "belief_kernel" not in name:
            continue
        ins = re.findall(r"/\*([0-9a-f]{4})\*/\s+([^;]*);", fn)
        ins = [(int(a, 16), t) for a, t in ins]
        addr = {a: i for i, (a, _) in enumerate(ins)}
        back = []
        for i, (_, t) in enumerate(ins):
            m = re.search(r"\bBRA(?:\.U)?\s+(?:!?U?P\d+,\s*)?0x([0-9a-f]+)", t)
            if m and addr.get(int(m.group(1), 16), i) < i:
                back.append((addr[int(m.group(1), 16)], i))
        total = mufu = 0
        for j, i in back:
            if any(j < j2 and i2 < i for j2, i2 in back):
                continue
            body = [t for _, t in ins[j:i + 1]]
            if any(re.search(r"\bBAR\b", t) for t in body):
                total += len(body)
                mufu += sum(1 for t in body if "MUFU" in t)
        res["polar_bp" if "polar_bp" in name else "polar"] = (total, mufu)
    return res


def pe_updates(n, T):
    m = int(np.log2(n))
    return ((2 * T - 1) * (m - 1) + 1) * n // 2


def sweep(model, ebnos):
    sim_ber(model, ebnos[:1], BS, 1, verbose=False)                       # warm-up: kernels, tables, buffers
    model._offset = 0
    t0 = time.perf_counter()
    _, bler = sim_ber(model, ebnos, BS, MAX_ITER, target_block_errs=TARGET, verbose=False)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return bler.numpy(), model._offset / wall


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bp.md"))
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bp_probe needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    print("card: %s, power limit %s, max SM clock %.0f MHz" % (name, power, clk / 1e6), flush=True)
    sass = loop_sass(dk.LIB_PATH)
    print("stage-loop SASS (instructions, MUFU):", sass, flush=True)
    rows = []
    for n, k in CODES:
        fp = po.rm_frozen_pos(n, n - k)
        tables = dk.code_tables(fp, n, dev)
        B = BYTES_IN // (4 * n)
        _, _, lg = dk.awgn_frontend(tables, B, ebno_mod.ebnodb2no(2.0, 2, k / n), 11)
        out = torch.empty((B, dk.words(n)), dtype=torch.int32, device=dev)
        for T in ITERS:
            for boxplus in (False, True):
                ms = median_ms(lambda: dk.belief_decode(lg, tables, T, boxplus, want_info=False, out_packed=out), args.reps)
                cws = B / ms * 1e3
                pe = pe_updates(n, T)
                ins, mufu = sass["polar_bp" if boxplus else "polar"]
                b_smem = SMS * SMEM_B_PER_CLK * clk / (24 * pe)
                b_issue = SMS * ISSUE_PER_CLK * clk * 32 / (ins / 2 * pe)
                b_mufu = SMS * MUFU_PER_CLK * clk * 32 / (mufu / 2 * pe) if mufu else float("inf")
                r = dict(n=n, k=k, T=T, arith="boxplus" if boxplus else "min-sum", B=B, ms=ms, cws=cws, fev=2 * pe * cws,
                         b_smem=b_smem, b_issue=b_issue, b_mufu=b_mufu)
                rows.append(r)
                print("n=%d T=%d %-7s %.3f ms  %.3e cw/s  %.3e f/s  bounds: smem %.3e issue %.3e mufu %.3e" % (
                    n, T, r["arith"], ms, cws, r["fev"], b_smem, b_issue, b_mufu), flush=True)
        del lg, out
    sw = []
    n, k = 1024, 512
    fp = po.rm_frozen_pos(n, n - k)
    rm_ebnos = np.array([2.0, 3.0, 4.0], dtype=np.float32)
    rm_decs = (("SC", lambda: SC_Dec(fp, n)), ("BP-20 boxplus", lambda: BP_Dec(fp, n)),
               ("BP-20 min-sum", lambda: BP_Dec(fp, n, cn_type="minsum")), ("SCL-8", lambda: SCL_Dec(fp, n, 8)))
    for dname, mk in rm_decs:
        bler, rate = sweep(System_AWGN_model(n, k, PolarEncoder(fp, n, None), mk(), seed=4242), rm_ebnos)
        sw.append(dict(code="(1024, 512) RM rule", dec=dname, ebnos=rm_ebnos, bler=bler, rate=rate))
        print(sw[-1], flush=True)
    k5, e5 = 100, 300
    enc = Polar5GEncoder(k5, e5)
    nr_ebnos = np.array([1.0, 2.0, 3.0], dtype=np.float32)

    def bp_minsum():
        d = Polar5GDecoder(enc, "BP")
        d._polar_dec = BP_Dec(enc._frozen_pos, enc.n_polar, cn_type="minsum")   # Polar5GDecoder's BP is boxplus
        return d
    nr_decs = (("SC", lambda: Polar5GDecoder(enc, "SC")), ("BP-20 boxplus", lambda: Polar5GDecoder(enc, "BP")),
               ("BP-20 min-sum", bp_minsum), ("SCL-8", lambda: Polar5GDecoder(enc, "SCL", list_size=8)))
    for dname, mk in nr_decs:
        bler, rate = sweep(System_AWGN_model(e5, k5, enc, mk(), seed=4242), nr_ebnos)
        sw.append(dict(code="(100, 300) 5G", dec=dname, ebnos=nr_ebnos, bler=bler, rate=rate))
        print(sw[-1], flush=True)

    lines = ["# Belief-propagation decoder (`polar_belief_decode_f32`)",
             "",
             "Measured with `python tools/bp_probe.py` on one %s at a %s power limit (max SM clock %.0f MHz, read in the "
             "same run)." % (name, power, clk / 1e6),
             "",
             "## Kernel throughput",
             "",
             "256 MB of logits per launch (B = 2^28 / 4n codewords, twice the L2), RM-rule codes, AWGN logits at 2 dB, packed "
             "output; CUDA-event median of %d launches after warm-up.  PE updates per codeword ((2T-1)(m-1)+1) n/2; two f "
             "evaluations each.  Bounds in codewords/s at the max SM clock over %d SMs: shared memory 24 B per PE update at "
             "%d B/clk/SM; issue %d warp instructions/clk/SM over the static SASS of the two stage loops (%d instructions "
             "min-sum, %d boxplus, of which %d MUFU); MUFU 16/clk/SM." % (
                 args.reps, SMS, SMEM_B_PER_CLK, ISSUE_PER_CLK, sass["polar"][0], sass["polar_bp"][0], sass["polar_bp"][1]),
             "",
             "| n | k | T | f | B | ms | codewords/s | f evaluations/s | smem bound | issue bound | MUFU bound | of the tightest |",
             "|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        tight = min(r["b_smem"], r["b_issue"], r["b_mufu"])
        which = "smem" if tight == r["b_smem"] else ("issue" if tight == r["b_issue"] else "MUFU")
        lines.append("| %d | %d | %d | %s | %d | %.3f | %.3e | %.3e | %.3e | %.3e | %s | %.0f %% (%s) |" % (
            r["n"], r["k"], r["T"], r["arith"], r["B"], r["ms"], r["cws"], r["fev"], r["b_smem"], r["b_issue"],
            "-" if r["b_mufu"] == float("inf") else "%.3e" % r["b_mufu"], 100 * r["cws"] / tight, which))
    lines += ["",
              "## BLER sweeps on the device loop",
              "",
              "`sim_ber` (on-device Monte-Carlo loop), batch %d, target %d block errors, at most %d iterations per point, "
              "after a one-iteration warm-up.  codewords/s = simulated codewords of the sweep over its wall time." % (
                  BS, TARGET, MAX_ITER),
              "",
              "| code | decoder | Eb/N0 (dB) | BLER per point | codewords/s |",
              "|---|---|---|---|---|"]
    for r in sw:
        lines.append("| %s | %s | %s | %s | %.3e |" % (r["code"], r["dec"], " / ".join("%g" % x for x in r["ebnos"]),
                                                      " / ".join("%.2e" % x for x in r["bler"]), r["rate"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))
    print("wrote", args.out)


if __name__ == "__main__":
    main()
