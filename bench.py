#!/usr/bin/env python
"""bench.py -- headline benchmark of the polar-code hot path on B200 (contract: see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): SC decoder, k=512 n=1024 RM-rule code, AWGN/BPSK at Eb/N0 = 4 dB,
batch B = 2^20 codewords per GPU (4 GiB of fp32 logits, larger than the 126 MB L2), synthetic, generated
on the device by polar_awgn_frontend.  One step = one decode of the whole batch.
  value : decoded information Gbit/s, whole job (all ranks), inputs resident in HBM, CUDA-event timed.
  e2e   : same metric through the reference's own boundary: SC_Dec.forward(cpu tensor [B,n]) -> cpu tensor [B,k] fp32
          (polar_sc.py:113-133; page-locked input, chunked H2D + decode + D2H inside the timed region); the bit-packed
          C-ABI side door (polar_sc_decode_host) and a pageable-input run are reported beside it.
  scl8  : the same numbers for SCL L=8 + CRC11 (configs[2], B = 2^18).
  link  : System_AWGN_model.forward (awgn_model.py:33-44) codewords/s: front end + decoder + API tensors.
  sweep : the BLER sweep (sim.py:79-133 through sim_ber_device) for configs[3] (SCL-32 n=2048, 9 points, 2^16 codewords per
          iteration over ALL ranks, target 1000 block errors, max 16 iterations) and for SC n=1024 (2^20 per iteration, 16
          iterations per point), batch sharded over the ranks (strong scaling), 4 x int64 all-reduce per iteration inside
          the timed region, with the per-iteration split.
--impl reference: the CPU restatement of the reference (oracle/libpolar_oracle.so, all host threads) on a
bounded sample per step (the reference itself is pure Python and cannot travel to the GPU box).
--dump-outputs DIR: after the timed steps, the decisions of the last step for a fixed, seeded sample of codewords
(dump_outputs), so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "polar-code-pytorch-sionna_b200")
for p in (ROOT, PKG, os.path.join(PKG, "x_run_sn_polar")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

N_CODE, K_CODE, EBNO_DB = 1024, 512, 4.0
SC_BATCH = 1 << 20
SCL_L, SCL_BATCH, SCL_CRC, SCL_EBNO_DB = 8, 1 << 18, "CRC11", 3.0


def frozen_set(n, k):
    """RM-rule frozen set of the reference (froze.py:4-16); golden fixture first (host-independent)."""
    path = os.path.join(ROOT, "tests", "golden", "frozen_sets.npz")
    key = "rm_%d_%d" % (n, k)
    if os.path.exists(path):
        d = np.load(path)
        if key in d:
            return d[key]
    from oracle import polar_oracle as po
    return po.rm_frozen_pos(n, n - k)


DUMP_ROWS = 8192        # 8192 x n=1024 fp32 = 32 MiB


def dump_rows(batch):
    """Batch indices of the codewords --dump-outputs writes: a fixed, seeded sample, the same for every run and build."""
    return np.sort(np.random.default_rng(0).choice(batch, size=min(batch, DUMP_ROWS), replace=False))


def dump_outputs(out_dir, rows, u_hat_bits):
    """DIR/u_hat.npy: the decisions u_hat[rows, 0:n] (frozen positions included) as fp32 0./1.;
    DIR/u_hat_rows.npy: the batch index of each of those rows, as float64."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "u_hat.npy"), np.asarray(u_hat_bits, dtype=np.float32))
    np.save(os.path.join(out_dir, "u_hat_rows.npy"), np.asarray(rows, dtype=np.float64))


_FULL_AFFINITY = None


def bind_to_gpu_numa_node(local_rank):
    """Several ranks per host: run this rank (and first-touch its pinned staging buffers) on the CPU socket the GPU's PCIe
    root hangs off, so the end-to-end leg of every rank streams from local DRAM.  Best effort; returns the node or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = None
        if all(hasattr(pr, a) for a in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
            bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        if bdf is None:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
            bdf = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
            bdf = bdf.decode() if isinstance(bdf, bytes) else bdf
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]                                            # nvml prints an 8-digit PCI domain, sysfs 4
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.windows = []          # [t0, t1] intervals (perf_counter) of the timed regions; only those samples count

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        inside = [r for (t, r) in self.rows if any(a - 0.05 <= t <= b + 0.15 for a, b in self.windows)]
        rows = inside if inside else [r for (_, r) in self.rows]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in rows:
            for i, nm in enumerate(names):
                if len(r) > 4 + i and r[4 + i].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_timed_regions": len(inside)}


# ----------------------------------------------------------------------------------------------------
def cpu_oracle_rate(kind, logits_np, frozen, L=0, seconds_hint=10.0):
    """Time the C oracle (all host threads) on a bounded sample; returns (cw/s, threads, n_codewords)."""
    from oracle import c_oracle as co
    co.build()
    if _FULL_AFFINITY and hasattr(os, "sched_setaffinity"):
        os.sched_setaffinity(0, _FULL_AFFINITY)             # the CPU leg uses every host core again (see bind_to_gpu_numa_node)
    thr = co.num_threads()
    t0 = time.perf_counter()
    if kind == "sc":
        co.sc_decode_full(logits_np, frozen)
    else:
        co.scl_decode_full(logits_np, frozen, L)
    dt = time.perf_counter() - t0
    return logits_np.shape[0] / dt, thr, logits_np.shape[0]


def run_reference(args):
    """--impl reference: CPU restatement of the reference path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import polar_oracle as po, c_oracle as co
    co.build()
    fp = frozen_set(N_CODE, K_CODE)
    fz = po.frozen_vec(fp, N_CODE)
    sample = 1 << 16
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import awgn_logits
    _, logits = awgn_logits(np.random.default_rng(1234), N_CODE, K_CODE, fp, sample, EBNO_DB)
    for _ in range(args.warmup):
        co.sc_decode_full(logits, fz)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        u_hat = co.sc_decode_full(logits, fz)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        rows = dump_rows(sample)
        dump_outputs(args.dump_outputs, rows, u_hat[rows])
    cws = sample * args.steps / dt
    val = cws * K_CODE / 1e9
    line = {"impl": "reference", "metric": "decoded_info_throughput_sc_n1024", "value": val, "unit": "Gbit/s",
            "codewords_per_s": cws, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "SC k=512 n=1024 AWGN BPSK Eb/N0=4dB (configs[1]); CPU restatement of the reference "
                                   "(oracle/polar_oracle.c, the Python reference cannot travel), %d-codeword sample per step" % sample},
            "cpu_baseline": {"value": val, "unit": "Gbit/s", "cores": co.num_threads(), "kind": "port",
                             "sample": "%d codewords per step x %d steps" % (sample, args.steps)},
            "e2e": {"value": val, "unit": "Gbit/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
KERNEL_SOURCES = {
    # files a kernel's translation unit is built from (csrc/Makefile): a capture is valid while these are unchanged
    "sc5_kernel<10>": ("polar_sc5.cu", "polar_common.cuh", "polar_warp.cuh", "polar_internal.h"),
    "scl3_kernel<10,8>": ("polar_scl3.cu", "polar_softplus.cuh", "polar_common.cuh", "polar_warp.cuh", "polar_internal.h"),
}


def source_stamp(kernel_key):
    """sha1 over the sources of one kernel: ncu-derived constants (instructions per codeword, DRAM bytes per launch) are
    only valid for the sources they were captured from (profiles/sc_counters.json carries the stamp of each capture)."""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(PKG, "csrc")
    for f in KERNEL_SOURCES[kernel_key]:
        h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_counters(kernel_key):
    """Counters captured by tools/refresh_counters.py for the CURRENT sources, else None (stale values are refused)."""
    p = os.path.join(ROOT, "profiles", "sc_counters.json")
    if not os.path.exists(p):
        return None, "no capture"
    d = json.load(open(p)).get(kernel_key)
    if not d:
        return None, "no capture"
    if d.get("source_stamp") != source_stamp(kernel_key):
        return None, "stale: captured for sources %s, current %s" % (d.get("source_stamp"), source_stamp(kernel_key))
    return d, "ncu capture of these sources (profiles/sc_counters.json)"


def run_sweep(kind, world, dev, sampler, barrier, max_over_ranks):
    """BLER sweep through the product's Monte-Carlo entry point (my_sn/sim.py::sim_ber_device; loop of sim.py:79-133,
    caller main.py:55-59).  Strong scaling: the per-iteration batch is split over the ranks; every iteration all-reduces
    the 4 counters (NCCL) in front of the on-device stop rules.  Timed wall clock, barrier + synchronize on both sides."""
    import torch
    from polar.enc import PolarEncoder
    from polar.polar_sc import SC_Dec
    from polar.polar_scl import SCL_Dec
    from z_sys_model.awgn_model import System_AWGN_model
    from my_sn.sim import sim_ber_device
    rank = int(os.environ.get("RANK", "0"))
    if kind == "scl32":
        n, k, total_bs, mc, tgt, name = 2048, 1024, 1 << 16, 16, 1000, "SCL L=32 k=1024 n=2048 (configs[3])"
        dec = lambda fp: SCL_Dec(fp, n, list_size=32)
    else:
        n, k, total_bs, mc, tgt, name = 1024, 512, 1 << 20, 16, None, "SC k=512 n=1024"
        dec = lambda fp: SC_Dec(fp, n)
    fp = frozen_set(n, k)
    ebnos = np.arange(0.0, 4.5, 0.5)
    bs = total_bs // world
    mk = lambda: System_AWGN_model(n, k, PolarEncoder(fp, n, None), dec(fp), seed=1234 + rank)
    sim_ber_device(mk(), ebnos[:2], bs, 2, target_block_errs=tgt, verbose=False)            # warm-up (allocators, NCCL)
    out = None
    times = []
    for rep in range(2):
        model = mk()
        stats = {}
        barrier()
        w0 = time.perf_counter()
        res = sim_ber_device(model, ebnos, bs, mc, target_block_errs=tgt, verbose=False, return_counters=True, stats=stats,
                             profile=(rep == 1))
        barrier()
        w1 = time.perf_counter()
        sampler.mark(w0, w1)
        times.append(max_over_ranks((w1 - w0) * 1e3))
        out = (res, stats)
    res, stats = out
    ms = min(times)
    counters = res[2]
    blocks = int(counters[:, 3].sum())                     # counted codewords over all ranks (the counters are all-reduced)
    return {"workload": "%s BLER sweep Eb/N0 0:0.5:4 dB, %d codewords per iteration over all ranks, max_mc_iter %d, target_block_errs %s"
                        % (name, total_bs, mc, tgt),
            "api": "my_sn.sim.sim_ber_device(System_AWGN_model(...)) -- what sim_ber / PlotBER.simulate / main.py run",
            "scaling": "strong", "n_gpus": world, "batch_per_rank": bs, "wall_ms": ms, "wall_ms_runs": times,
            "simulated_codewords": blocks, "codewords_per_s": blocks / (ms * 1e-3), "info_gbit_per_s": blocks / (ms * 1e-3) * k / 1e9,
            "iterations_counted": int(res[4].sum()), "iterations_queued": stats.get("queued"), "decoder_launches": stats.get("groups"),
            "bler": [float(v) for v in res[1]], "split_us_per_iteration": stats.get("split_us"),
            "collective": "ncclAllReduce of the group's n_items x 4 int64 counters, one per decoder launch" if world > 1 else "none (one rank)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=SC_BATCH, help="SC codewords per GPU per step")
    ap.add_argument("--skip-scl", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--skip-link", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the SC decisions of the last timed step (rank 0, seeded sample of %d codewords) to DIR" % DUMP_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import d_kernels as dk
    from oracle import polar_oracle as po      # checker + cpu_baseline leg only
    from polar.polar_sc import SC_Dec

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    global _FULL_AFFINITY
    _FULL_AFFINITY = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner (and NCCL_DEBUG output) to fd 1 while the
        # communicator is created, so fd 1 points at stderr until the first collective is through
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    n, k, B = N_CODE, K_CODE, args.batch
    fp = frozen_set(n, k)
    tables = dk.code_tables(fp, n, dev)
    no = po.ebnodb2no(EBNO_DB, 2, k / n)
    nw = dk.words(n)
    # ---- inputs resident in HBM before timing (front-end kernel, seed 1234 + rank) --------------------
    u_tx, _, logits = dk.awgn_frontend(tables, B, no, 1234 + rank)
    u_hat = torch.empty((B, nw), dtype=torch.int32, device=dev)
    stream = dk.stream_ptr(dev)
    lib = dk.lib()

    def sc_step():
        dk.check(lib.polar_sc_decode_f32(dk.ptr(logits), dk.ptr(tables.frozen_mask), n, B, dk.ptr(u_hat), None, None, 0, stream))

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # runs through every timed region of this process
    for _ in range(args.warmup):
        sc_step()
    barrier()
    launches0 = dk.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_all0, t_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    t_all0.record()
    for a, b in evs:
        a.record(); sc_step(); b.record()
    t_all1.record()
    barrier()
    sampler.mark(w0, time.perf_counter())
    launches = dk.launch_count() - launches0
    total_ms = max_over_ranks(t_all0.elapsed_time(t_all1))
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))      # one launch per step: the SC kernel itself
    ms_per_step = total_ms / args.steps
    cws = world * B / (ms_per_step * 1e-3)
    value = cws * k / 1e9
    if args.dump_outputs and rank == 0:
        rows = dump_rows(B)
        words = u_hat[torch.from_numpy(rows).to(dev)].cpu().numpy()
        dump_outputs(args.dump_outputs, rows, np.unpackbits(words.view(np.uint8), axis=-1, bitorder="little")[:, :n])

    # ---- same decode writing the reference's API tensor [B,k] fp32 as well (SURVEY 8d C2: "report both") -----
    u_api = torch.empty((B, k), dtype=torch.float32, device=dev)

    def sc_api_step():
        dk.check(lib.polar_sc_decode_f32(dk.ptr(logits), dk.ptr(tables.frozen_mask), n, B, None, dk.ptr(u_api), dk.ptr(tables.info_pos), k, stream))
    sc_api_step()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    api_steps = max(3, min(args.steps, 10))
    a.record()
    for _ in range(api_steps):
        sc_api_step()
    b.record()
    barrier()
    api_ms = max_over_ranks(a.elapsed_time(b) / api_steps)
    api_tensor = {"value": world * B / (api_ms * 1e-3) * k / 1e9, "unit": "Gbit/s", "codewords_per_s": world * B / (api_ms * 1e-3),
                  "ms_per_step": api_ms, "output": "[B,k] fp32 0./1. (what SC_Dec.forward returns; %d MiB per step) instead of the "
                  "bit-packed decisions (%d MiB)" % (B * k * 4 >> 20, B * nw * 4 >> 20),
                  "matches_packed": bool(torch.equal(u_api[:4096], dk.unpack_info(u_hat[:4096], tables.info_pos, n)))}
    launches += api_steps + 1

    # ---- parity spot check in the same run (bit-exact vs the oracle on a slice; BLER sanity) ------------
    parity = None
    if rank == 0:
        from oracle import c_oracle as co
        co.build()
        m_chk = 4096
        ref = co.sc_decode_full(logits[:m_chk].cpu().numpy(), po.frozen_vec(fp, n))
        got = np.unpackbits(u_hat[:m_chk].cpu().numpy().view(np.uint8), axis=-1, bitorder="little")[:, :n]
        cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        dk.count_errors_packed(u_tx, u_hat, tables.info_mask, n, cnt)
        c = cnt.cpu().numpy()
        parity = {"bit_exact_vs_oracle": bool(np.array_equal(got, ref)), "checked_codewords": m_chk,
                  "bler": float(c[1]) / B, "ber": float(c[0]) / (B * k),
                  "full_batch_parity": "tests/test_gpu_fullsize.py (all 2^20 codewords, -m gpu)"}

    # ---- end to end through the reference's boundary: SC_Dec.forward(cpu tensor) -> cpu tensor -----------
    e2e = None
    if not args.skip_e2e:
        sc_mod = SC_Dec(fp, n, device=dev)
        h_logits = torch.empty((B, n), dtype=torch.float32, pin_memory=True)
        h_logits.copy_(logits)
        ref_info = u_api[:4096].cpu()

        def timed(fn, steps):
            for _ in range(3):                                     # warm-up: staging buffers, and torch's page-locked
                r = fn()                                           # allocator has to have BOTH result buffers it ping-pongs
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                r = fn()
            torch.cuda.synchronize()
            return max_over_ranks((time.perf_counter() - t0) * 1e3 / steps), r
        e2e_steps = max(3, min(args.steps, 5))
        w0 = time.perf_counter()
        mod_ms, out = timed(lambda: sc_mod(h_logits), e2e_steps)
        sampler.mark(w0, time.perf_counter())
        ok = bool(out.device.type == "cpu" and out.shape == (B, k) and torch.equal(out[:4096], ref_info))
        e2e = {"value": world * B / (mod_ms * 1e-3) * k / 1e9, "unit": "Gbit/s", "h2d_bytes_per_step": B * n * 4,
               "d2h_bytes_per_step": B * k * 4, "ms_per_step": mod_ms, "codewords_per_s": world * B / (mod_ms * 1e-3),
               "api": "SC_Dec.forward(cpu fp32 tensor [B,n], page-locked) -> cpu fp32 tensor [B,k] (x_run_sn_polar/polar/polar_sc.py; "
                      "C ABI polar_sc_decode_host_f32: 32 MB chunks (128 MB when the input is pageable and staged), H2D / decode / D2H on two streams)",
               "matches_device_path": ok}
        del out
        # the bit-packed C-ABI side door (round 1's e2e number): 32x less D2H
        h_out = torch.empty((B, nw), dtype=torch.int32, pin_memory=True)
        mask_np = tables.mask_np
        pk_ms, _ = timed(lambda: dk.check(lib.polar_sc_decode_host(h_logits.data_ptr(), mask_np.ctypes.data, n, B, h_out.data_ptr(), local)),
                         e2e_steps)
        e2e["packed_c_abi"] = {"value": world * B / (pk_ms * 1e-3) * k / 1e9, "unit": "Gbit/s", "ms_per_step": pk_ms,
                               "d2h_bytes_per_step": B * nw * 4, "api": "polar_sc_decode_host (bit-packed decisions)",
                               "matches_device_path": bool(torch.equal(h_out[:4096], u_hat[:4096].cpu()))}
        del h_out
        # pageable input (a plain torch CPU tensor): staged through page-locked buffers by host threads
        Bp = min(B, 1 << 18)
        pg = torch.empty((Bp, n), dtype=torch.float32)
        pg.copy_(h_logits[:Bp])
        pg_ms, outp = timed(lambda: sc_mod(pg), 3)
        e2e["pageable_input"] = {"value": world * Bp / (pg_ms * 1e-3) * k / 1e9, "unit": "Gbit/s", "ms_per_step": pg_ms, "batch": Bp,
                                 "api": "SC_Dec.forward(pageable cpu tensor)", "matches_device_path": bool(torch.equal(outp[:4096], ref_info))}
        del h_logits, pg, outp
    del u_api

    peaks, peak_src = measured_peaks()
    # ---- link level: System_AWGN_model.forward (front end + decoder + API tensors), awgn_model.py:33-44 ----
    link = None
    if not args.skip_link:
        from polar.enc import PolarEncoder
        from z_sys_model.awgn_model import System_AWGN_model
        Bl = 1 << 18
        model = System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n, device=dev), device=dev, seed=77 + rank)
        for _ in range(4):
            model(Bl, EBNO_DB)
        barrier()
        l0 = dk.launch_count()
        reps = 10
        evl = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evl:
            a.record()
            bits, bits_hat = model(Bl, EBNO_DB)
            b.record()
        barrier()
        launches += dk.launch_count() - l0
        per_call = [a.elapsed_time(b) for a, b in evl]
        ms = max_over_ranks(float(np.median(per_call)))          # median: torch's allocator occasionally returns memory mid-loop
        ms_mean = max_over_ranks(float(np.mean(per_call)))
        link = {"metric": "link_model_throughput_sc_n1024", "codewords_per_s": world * Bl / (ms * 1e-3),
                "value": world * Bl / (ms * 1e-3) * k / 1e9, "unit": "Gbit/s", "ms_per_step": ms, "ms_per_step_mean": ms_mean, "batch": Bl,
                "api": "System_AWGN_model.forward(batch_size, ebno_db) -> (bits [B,k], bits_hat [B,k]) fp32 device tensors "
                       "(polar_awgn_frontend + sc5_kernel + 2 unpack kernels per call)",
                "bler": float((bits != bits_hat).any(dim=1).float().mean().item())}
        del bits, bits_hat, model

    # ---- SCL L=8 + CRC11 (configs[2]) ------------------------------------------------------------------
    scl = None
    if not args.skip_scl:
        from my_sn.fec.crc import CRCEncoder
        from my_sn.fec.polar.dec import SCL_Dec as SclCrcDec
        Bs = SCL_BATCH
        crc_chk = CRCEncoder(SCL_CRC, k)                       # validity check spans all k decoder outputs (dec.py:508-516)
        crc = CRCEncoder(SCL_CRC, k - crc_chk.crc_length)      # generator for the payload
        rows = torch.from_numpy(crc_chk.syndrome_rows(tables.info_pos_np, n).view(np.int32).copy()).to(dev)
        no_s = po.ebnodb2no(SCL_EBNO_DB, 2, k / n)
        # payload + CRC parity -> polar codeword -> channel, all on the device (untimed set-up)
        payload = torch.randint(0, 2, (Bs, k - crc.crc_length), device=dev, dtype=torch.float32)
        bits = crc(payload)
        cw = dk.encode_f32(bits, tables)
        lg = dk.qpsk_awgn_llr(cw, no_s, 4321 + rank)
        best = torch.empty((Bs, nw), dtype=torch.int32, device=dev)
        need = int(lib.polar_scl_workspace_bytes(n, SCL_L, Bs))
        ws = torch.empty(max(need, 256) + 256, dtype=torch.uint8, device=dev)
        ws_ptr = (ws.data_ptr() + 255) // 256 * 256

        def scl_step():
            dk.check(lib.polar_scl_decode(dk.ptr(lg), dk.ptr(tables.frozen_mask), n, SCL_L, Bs, dk.ptr(best), None, None, k,
                                          None, None, dk.ptr(rows), crc.crc_length, ws_ptr, need, stream))
        scl_steps = max(3, min(args.steps, 5))
        for _ in range(2):
            scl_step()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = dk.launch_count()
        w0 = time.perf_counter()
        a.record()
        for _ in range(scl_steps):
            scl_step()
        b.record()
        barrier()
        sampler.mark(w0, time.perf_counter())
        launches += dk.launch_count() - l0
        scl_ms = max_over_ranks(a.elapsed_time(b) / scl_steps)
        scl_cws = world * Bs / (scl_ms * 1e-3)
        cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        full = torch.zeros((Bs, n), dtype=torch.float32, device=dev)
        full[:, tables.info_pos.long()] = bits
        txu = dk.pack_bits(full)
        dk.count_errors_packed(txu, best, tables.info_mask, n, cnt)
        c = cnt.cpu().numpy()
        del full
        sm_clk_now = 1965.0
        cnts, cnts_src = ncu_counters("scl3_kernel<10,8>")
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        issue_peak = sms * 4 * sm_clk_now * 1e6
        roof = {"bound": "issue", "unit": "warp-instr/s", "peak": issue_peak, "achieved": None, "frac": None, "traffic": None,
                "counters": cnts_src,
                "note": "the list decoder is instruction bound, not HBM bound (algorithmic bytes 4n + k/8 per codeword = %.4f of HBM "
                        "peak at this rate): achieved = codewords/s x warp instructions per codeword (ncu smsp__inst_executed / batch), "
                        "peak = SMs x 4 schedulers x SM clock" % (scl_cws / world * (4 * n + k / 8) / 1e9 / peaks["hbm_gbs"])}
        if cnts:
            ach = scl_cws / world * cnts["warp_instr_per_codeword"]
            roof.update(achieved=ach, frac=ach / issue_peak, traffic=cnts.get("dram_bytes_per_launch"),
                        warp_instr_per_codeword=cnts["warp_instr_per_codeword"])
        scl = {"metric": "decoded_info_throughput_scl8_crc11_n1024", "value": scl_cws * k / 1e9, "unit": "Gbit/s",
               "codewords_per_s": scl_cws, "ms_per_step": scl_ms, "batch": Bs, "ebno_db": SCL_EBNO_DB,
               "bler": float(c[1]) / Bs, "workload": "SCL L=8 k=512 (501+CRC11) n=1024 CRC-aided selection, batch 256K (configs[2])",
               "kernel": "scl3_kernel<10,8,...> (polar_scl3.cu)", "roofline": roof}
        if not args.skip_e2e:
            mod = SclCrcDec(fp, n, SCL_L, crc_degree=SCL_CRC, cn_type="minsum", device=dev)
            h_lg = torch.empty((Bs, n), dtype=torch.float32, pin_memory=True)
            h_lg.copy_(lg)
            want = dk.unpack_info(best[:2048], tables.info_pos, n).cpu()
            for _ in range(3):
                out = mod(h_lg)
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                out = mod(h_lg)
            torch.cuda.synchronize()
            ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / 3)
            scl["e2e"] = {"value": world * Bs / (ms * 1e-3) * k / 1e9, "unit": "Gbit/s", "h2d_bytes_per_step": Bs * n * 4,
                          "d2h_bytes_per_step": Bs * k * 4 + Bs * SCL_L * 8, "ms_per_step": ms,
                          "api": "my_sn.fec.polar.dec.SCL_Dec(crc_degree='CRC11').forward(cpu tensor) -> cpu tensor [B,k] fp32 "
                                 "(polar_scl_decode_host_f32)",
                          "matches_device_path": bool(torch.equal(out[:2048], want))}
            if not scl["e2e"]["matches_device_path"]:
                full_want = dk.unpack_info(best, tables.info_pos, n).cpu()
                badrows = (out != full_want).any(dim=1).nonzero().flatten()
                dev_mod = mod(lg).cpu()
                scl["e2e"]["debug"] = {"bad_rows": int(badrows.numel()), "first": badrows[:8].tolist(),
                                       "device_module_equals_packed": bool(torch.equal(dev_mod, full_want)),
                                       "host_equals_device_module": bool(torch.equal(dev_mod, out))}
            del h_lg, out
        if rank == 0 and not args.skip_cpu:
            smp = 16384
            rate, thr, cnt_cw = cpu_oracle_rate("scl", lg[:smp].cpu().numpy(), po.frozen_vec(fp, n), SCL_L)
            scl["cpu_baseline"] = {"value": rate * k / 1e9, "unit": "Gbit/s", "codewords_per_s": rate, "cores": thr, "kind": "port",
                                   "sample": "first %d codewords of the GPU batch, C restatement (oracle/polar_oracle.c)" % cnt_cw}
        del lg, cw, bits, payload, best, ws

    # ---- BLER sweeps (strong scaling over the ranks) ---------------------------------------------------------
    sweep = None
    if not args.skip_sweep:
        del logits, u_hat, u_tx
        torch.cuda.empty_cache()
        l0 = dk.launch_count()
        sweep = {"scl32_n2048": run_sweep("scl32", world, dev, sampler, barrier, max_over_ranks),
                 "sc_n1024": run_sweep("sc", world, dev, sampler, barrier, max_over_ranks)}
        launches += dk.launch_count() - l0
        logits = None

    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    bytes_per_cw = 4 * n + k // 8           # SURVEY 8(d): fp32 logits in, bit-packed decisions out (k info bits)
    achieved = B * bytes_per_cw / (kern_ms * 1e-3) / 1e9
    cpu = None
    if not args.skip_cpu:
        smp = min(B, 1 << 20)
        if logits is None:
            _, _, logits = dk.awgn_frontend(tables, smp, no, 1234 + rank)
        rate, thr, cnt_cw = cpu_oracle_rate("sc", logits[:smp].cpu().numpy(), po.frozen_vec(fp, n))
        cpu = {"value": rate * k / 1e9, "unit": "Gbit/s", "codewords_per_s": rate, "cores": thr, "kind": "port",
               "sample": "first %d codewords of the GPU batch, C restatement of the reference (oracle/polar_oracle.c); "
                         "the Python reference itself measured 3270 cw/s on 8 vCPU (BASELINE.md)" % cnt_cw}
    # SURVEY 8(d): the other candidate bounds next to HBM.  Instruction count / DRAM traffic come from an ncu capture of the
    # CURRENT sources (profiles/sc_counters.json, stamped with a hash of csrc/); a stale capture is refused, not reused.
    sm_clk = (clocks or {}).get("sm_mhz") or 1965.0
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    cw_rate_gpu = B / (kern_ms * 1e-3)
    issue_peak = sms * 4 * sm_clk * 1e6  # one warp instruction per scheduler and cycle
    cnts, cnts_src = ncu_counters("sc5_kernel<10>")
    traffic = None
    other_bounds = {"counters": cnts_src}
    if cnts and B == (1 << 20):
        traffic = cnts.get("dram_bytes_per_launch")
        wi = cnts["warp_instr_per_codeword"]
        other_bounds["issue"] = {"achieved": cw_rate_gpu * wi, "peak": issue_peak, "unit": "warp-instr/s",
                                 "frac": cw_rate_gpu * wi / issue_peak, "warp_instr_per_codeword": wi}
        if traffic:
            other_bounds["dram_actual"] = {"achieved": traffic / (kern_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                           "frac": traffic / (kern_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
    line = {
        "metric": "decoded_info_throughput_sc_n1024", "value": value, "unit": "Gbit/s", "codewords_per_s": cws,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "SC k=512 n=1024 RM-rule code, AWGN BPSK Eb/N0=4dB, batch %d codewords per GPU (configs[1])" % B,
                   "l2": "inputs (%.1f GiB per GPU) larger than L2, no flush needed" % (B * n * 4 / 2 ** 30),
                   "parallelism": "batch sharded over %d rank(s), no data-path collective" % world,
                   "numa_node_rank0": numa},
        "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_src,
                     "kernel": "sc5_kernel<10,6> (polar_sc5.cu)", "kernel_ms": kern_ms, "bytes_per_codeword": bytes_per_cw,
                     "other_bounds": other_bounds,
                     "note": "algorithmic bytes = 4n + k/8 per codeword; achieved = B x 4160 B / mean CUDA-event time of the kernel "
                             "launches of the timed region (DESIGN.md 4.1)"},
        "api_tensor_output": api_tensor, "link": link, "sweep": sweep,
        "cpu_baseline": cpu, "parity": parity, "scl8": scl,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
