"""5G NR polar codes through the fused AWGN link model: the front end `polar_nr5g_awgn_frontend` alone, and BLER sweeps of
four rate-matched codes on the three Monte-Carlo paths a user can take.

Front end: 2^20 codewords per launch, CUDA-event median of REPS launches after warm-up; bytes written = 4 e (logits) +
4 words(n) (payload + CRC words) per codeword, over kernel time, against the HBM copy bandwidth measured in the same run
(device-to-device copy of 4 GiB: 8 GiB moved).  The plain power-of-two front end of the mother code is timed alongside.

Sweeps (SC, SCL-8, hybSCL-8 of Polar5GDecoder; target 1000 block errors, at most MAX_ITER iterations of BS codewords per
point): wall time and counted codewords/s of
  - sim_ber (on-device loop, the default),
  - sim_ber(on_device=False) (fused front end, host loop),
  - fused=False (the layer-by-layer torch composition, host loop), for the (100, 300) code only.

  python tools/nr5g_probe.py [--out profiles/r04_nr5g_link.md] [--reps 20]"""
import argparse
import os
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
from my_sn.fec.polar.enc import Polar5GEncoder
from my_sn.fec.polar.dec import Polar5GDecoder
from my_sn.sim import sim_ber
from my_sn.trans import ebno as ebno_mod
from z_sys_model.awgn_model import System_AWGN_model

# Eb/N0 grids: SCL-8 BLER from ~1e-1 down to where the iteration cap, not the error target, ends the point
CODES = ((64, 128, "none", (2.0, 3.0, 4.0, 5.0)), (100, 300, "puncturing", (1.0, 2.0, 3.0, 4.0)),
         (200, 400, "shortening", (1.0, 2.0, 3.0, 4.0)), (300, 1088, "repetition", (0.5, 1.0, 1.5, 2.0)))
DECODERS = ("SC", "SCL", "hybSCL")
B_FE, BS, MAX_ITER, TARGET = 1 << 20, 1 << 14, 100, 1000
LAYER_CODE, LAYER_MAX_ITER = (100, 300), 30


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


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


def hbm_copy_gbs(reps):
    src = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    ms = median_ms(lambda: dst.copy_(src), reps)
    del src, dst
    return 2 * 4 * (1 << 30) / ms / 1e6


def counting(model):
    """Count the codewords a host loop simulates (forward calls x batch)."""
    model.n_cw = 0
    fwd = model.forward

    def f(batch_size, ebno_db):
        model.n_cw += int(batch_size)
        return fwd(batch_size, ebno_db)
    model.forward = f
    return model


def sweep(enc, kind, path, ebnos):
    k, e = enc.k, enc.n
    model = System_AWGN_model(e, k, enc, Polar5GDecoder(enc, kind, list_size=8), fused=path != "layers", seed=4242)
    counting(model)
    mi = LAYER_MAX_ITER if path == "layers" else MAX_ITER
    t0 = time.perf_counter()
    ber, bler = sim_ber(model, ebnos, BS, mi, target_block_errs=TARGET, verbose=False, on_device=path == "device")
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    cw = model._offset if path == "device" else model.n_cw
    return dict(wall=wall, cw=cw, bler=bler.numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_nr5g_link.md"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "nr5g_probe needs a CUDA device"
    dev = torch.device("cuda", 0)
    gpu = card()
    print("card:", gpu, flush=True)
    peak = hbm_copy_gbs(args.reps)
    print("HBM copy %.0f GB/s" % peak, flush=True)
    fe = []
    for k, e, rm, _ in CODES:
        enc = Polar5GEncoder(k, e)
        plan = enc.frontend_plan(dev)
        no = ebno_mod.ebnodb2no(1.0, 2, k / e)
        u = torch.empty((B_FE, dk.words(plan.n)), dtype=torch.int32, device=dev)
        lg = torch.empty((B_FE, e), dtype=torch.float32, device=dev)
        ms = median_ms(lambda: dk.nr5g_awgn_frontend(plan, B_FE, no, 7, 0, out=(u, lg)), args.reps)
        tables = dk.code_tables(enc.frozen_pos, plan.n, dev)
        lg_p = torch.empty((B_FE, plan.n), dtype=torch.float32, device=dev)
        ms_p = median_ms(lambda: dk.awgn_frontend(tables, B_FE, no, 7, 0, out=(u, lg_p)), args.reps)
        del lg, lg_p, u
        by = B_FE * (4 * e + 4 * dk.words(plan.n))
        by_p = B_FE * (4 * plan.n + 4 * dk.words(plan.n))
        r = dict(k=k, e=e, n=plan.n, rm=rm, ms=ms, gbs=by / ms / 1e6, ms_p=ms_p, gbs_p=by_p / ms_p / 1e6)
        fe.append(r)
        print("front end k=%d E=%d n=%d: %.3f ms, %.0f GB/s (%.0f %% of copy); plain n=%d: %.3f ms, %.0f GB/s" % (
            k, e, plan.n, ms, r["gbs"], 100 * r["gbs"] / peak, plan.n, ms_p, r["gbs_p"]), flush=True)
    sw = []
    for k, e, rm, ebnos in CODES:
        enc = Polar5GEncoder(k, e)
        ebnos = np.array(ebnos, dtype=np.float32)
        for kind in DECODERS:
            paths = ("device", "host") + (("layers",) if (k, e) == LAYER_CODE else ())
            for p in paths:                                                # warm-up: kernels, tables, buffers, layers
                m = System_AWGN_model(e, k, enc, Polar5GDecoder(enc, kind, list_size=8), fused=p != "layers", seed=1)
                sim_ber(m, ebnos[:1], BS, 1, verbose=False, on_device=p == "device")
            res = {p: sweep(enc, kind, p, ebnos) for p in paths}
            same = bool(np.array_equal(res["device"]["bler"], res["host"]["bler"]))
            for p in paths:
                r = res[p]
                sw.append(dict(k=k, e=e, rm=rm, kind=kind, path=p, wall=r["wall"], cw=r["cw"], rate=r["cw"] / r["wall"],
                               bler=r["bler"], same=same, ebnos=ebnos))
                print("k=%d E=%d %-6s %-6s wall %.3f s  %d cw  %.3e cw/s  BLER %s  device==host %s" % (
                    k, e, kind, p, r["wall"], r["cw"], r["cw"] / r["wall"], np.array2string(r["bler"], precision=3), same),
                    flush=True)
    lines = ["# 5G NR polar codes in the fused AWGN link model",
             "",
             "Measured with `python tools/nr5g_probe.py` on one %s (name, power limit)." % gpu,
             "",
             "## Front end alone (`polar_nr5g_awgn_frontend`)",
             "",
             "%d codewords per launch, CUDA-event median of %d launches after warm-up.  Bytes = 4 e + 4 words(n) per codeword "
             "written (logits and payload + CRC words; the rate-matched codeword output is off).  HBM copy bandwidth measured "
             "in the same run (4 GiB device-to-device copy): %.0f GB/s.  The plain front end (`polar_awgn_frontend`) of the "
             "mother code, same codewords, is shown for comparison." % (B_FE, args.reps, peak),
             "",
             "| k | E | n_polar | rate matching | ms | GB/s written | of copy BW | plain n_polar ms | plain GB/s |",
             "|---|---|---|---|---|---|---|---|---|"]
    for r in fe:
        lines.append("| %d | %d | %d | %s | %.3f | %.0f | %.0f %% | %.3f | %.0f |" % (
            r["k"], r["e"], r["n"], r["rm"], r["ms"], r["gbs"], 100 * r["gbs"] / peak, r["ms_p"], r["gbs_p"]))
    lines += ["",
              "## BLER sweeps",
              "",
              "Batch %d, target %d block errors, at most %d iterations per point (%d on the layer path), "
              "early stop at an error-free point.  `device` = `sim_ber` (on-device loop, the default), `host` = "
              "`sim_ber(on_device=False)` (fused front end, host loop), `layers` = `fused=False` (torch layer composition). "
              "Wall time of the whole sweep after a warm-up run; codewords = counted codewords of all points. "
              "`same` = device and host loop give identical BLER." % (
                  BS, TARGET, MAX_ITER, LAYER_MAX_ITER),
              "",
              "| k | E | rate matching | decoder | path | Eb/N0 (dB) | wall s | codewords | codewords/s | BLER per point | same |",
              "|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in sw:
        lines.append("| %d | %d | %s | %s | %s | %s | %.3f | %d | %.3e | %s | %s |" % (
            r["k"], r["e"], r["rm"], r["kind"], r["path"], " / ".join("%g" % x for x in r["ebnos"]), r["wall"], r["cw"], r["rate"],
            " / ".join("%.2e" % x for x in r["bler"]), "yes" if r["same"] else "no"))
    lines.append("")
    for r in sw:
        if r["path"] == "device":
            h = [x for x in sw if x["path"] == "host" and (x["k"], x["e"], x["kind"]) == (r["k"], r["e"], r["kind"])][0]
            lines.append("- k=%d, E=%d, %s: device loop %.2fx the host loop in codewords/s." % (
                r["k"], r["e"], r["kind"], r["rate"] / h["rate"]))
            la = [x for x in sw if x["path"] == "layers" and (x["k"], x["e"], x["kind"]) == (r["k"], r["e"], r["kind"])]
            if la:
                lines[-1] += "  %.1fx the layer path (`fused=False`)." % (r["rate"] / la[0]["rate"])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))
    print("wrote", args.out)


if __name__ == "__main__":
    main()
