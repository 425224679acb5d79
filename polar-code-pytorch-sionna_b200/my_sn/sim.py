"""Monte-Carlo BER/BLER loop with the reference call surface (my_sn/sim.py:4-140).

Differences that matter on B200: the bit/block error counts of an iteration are produced by one
fused kernel (`polar_count_errors_f32`) into a device counter pair and read back once per iteration
(the stop rules of sim.py:107-133 need them on the host); when `torch.distributed` is initialised the
four counters are combined with one 4 x int64 all-reduce per iteration so every rank takes the same
stop decisions (SURVEY 8e).  `mc_fun` is then expected to simulate its shard (batch_size is the
per-rank batch).  When `mc_fun` is the fused AWGN link model, `sim_ber` hands over to `sim_ber_device`, which keeps
the whole loop -- including the stop rules -- on the device (SURVEY 8f row N1)."""
import time

import numpy as np
import torch as tc

import d_kernels as dk


def hard_decisions(llr):
  return tc.where(llr > 0, 1., 0.)


def _count(b, b_hat):
  """(bit errors, block errors) between two 0/1 tensors (sim.py:7-18) as Python ints."""
  if b.is_cuda or b_hat.is_cuda:
    dev = b.device if b.is_cuda else b_hat.device
    counters = tc.zeros(2, dtype=tc.int64, device=dev)
    dk.count_errors_f32(b, b_hat, counters)
    c = counters.cpu()
    return int(c[0]), int(c[1])
  raise RuntimeError("polar_b200: count_errors needs CUDA tensors (no CPU fallback)")


def count_errors(b, b_hat):
  """Number of bit errors (sim.py:15-18); returns a 0-dim int64 tensor like the reference."""
  return tc.tensor(_count(b, b_hat)[0], dtype=tc.int64)


def count_block_errors(b, b_hat):
  """Number of rows with at least one differing element (sim.py:7-14)."""
  return tc.tensor(_count(b, b_hat)[1], dtype=tc.int64)


def _dist():
  import torch.distributed as dist
  return dist if (dist.is_available() and dist.is_initialized()) else None


def _device_loop_ok(mc_fun, soft_estimates, count_fn):
  """The on-device loop applies to link models that provide the `device_frontend` hook (fused AWGN / BEC front end)
  together with a decoder that has the packed fast path."""
  return (count_fn is None and not soft_estimates and getattr(mc_fun, "fused", False)
          and callable(getattr(mc_fun, "device_frontend", None))
          and not getattr(mc_fun, "cw_estimates", True) and hasattr(getattr(mc_fun, "decoder", None), "decode_packed")
          and tc.cuda.is_available())


class SweepPlanner:
  """Which (SNR point, iteration) work items will the sequential loop of sim.py:79-133 run next?

  The device loop packs several items into one decoder launch (a per-rank batch of a few thousand codewords leaves the
  last wave of a persistent kernel half empty) and keeps a second group queued behind the first.  An item that the
  sequential loop would not have run at its position -- a point stopped earlier or later than planned -- is ignored by
  the control kernel together with everything queued behind it, so a wrong plan only costs time, never a result.  The
  planner therefore commits to a stop only when it is certain at ~3 sigma: from this point's counters so far, else from
  bounds chained from the last finished point (error rates fall with Eb/N0: upper bound = the previous point's rate,
  lower bound = `damp` times its lower bound).  Where the stop is uncertain the group ends at the earliest possible stop
  and the next group waits for the counters.

  State of a plan: (point, iterations counted at it, lower / upper bound of its (bit, block) error counts so far)."""

  def __init__(self, n_points, target_bit_errs, target_block_errs, max_mc_iter, per_iter_max, damp=0.3):
    self.P = int(n_points)
    self.targets = (target_bit_errs, target_block_errs)
    self.max_iter = int(max_mc_iter)
    self.damp = float(damp)
    # per-iteration (bit, block) error rate bounds of the last finished point; before the first: the most a batch can hold
    self.prev_hi = tuple(float(v) for v in per_iter_max)
    self.prev_lo = tuple(float(v) * self.damp for v in per_iter_max)

  def finished_point(self, iters, bit_errs, block_errs):
    """Counters of the point that just finished: the next points' rates are bounded by them."""
    if iters > 0:
      r = (bit_errs / iters, block_errs / iters)
      self.prev_hi = tuple(v + 3.0 * (v / iters) ** 0.5 + 1.0 / iters for v in r)
      self.prev_lo = tuple(max(v - 3.0 * (v / iters) ** 0.5 - 1.0 / iters, 0.0) * self.damp for v in r)

  def _stop_range(self, cum_lo, cum_hi, lo, hi, rem):
    """(earliest possible, surely reached) number of further iterations until a target stops the point, both <= rem."""
    r_lo = r_hi = rem
    for t in range(2):
      tgt = self.targets[t]
      if tgt is None:
        continue
      for r in range(1, rem + 1):
        if cum_hi[t] + r * hi[t] + 3.0 * (r * hi[t]) ** 0.5 + 1.0 >= tgt:
          r_lo = min(r_lo, r)
          break
      for r in range(1, rem + 1):
        if cum_lo[t] + r * lo[t] - 3.0 * (r * lo[t]) ** 0.5 - 1.0 >= tgt:
          r_hi = min(r_hi, r)
          break
    return r_lo, max(r_hi, r_lo)

  def plan(self, state, gmax):
    """state = (point, iters, cum_lo, cum_hi) -> (items: list of point indices, state after them or None when the last
    item may or may not stop its point, "done" when the plan reaches the end of the sweep)."""
    p, it, cum_lo, cum_hi = state
    items = []
    chain_lo, chain_hi = self.prev_lo, self.prev_hi
    while len(items) < gmax and p < self.P:
      if it > 0:      # this point's own counters bound its rate
        lo = tuple(max(c / it - 3.0 * (c / it / it) ** 0.5 - 1.0 / it, 0.0) for c in cum_lo)
        hi = tuple(c / it + 3.0 * (c / it / it) ** 0.5 + 1.0 / it for c in cum_hi)
      else:
        lo, hi = chain_lo, chain_hi
      rem = self.max_iter - it
      r_lo, r_hi = self._stop_range(cum_lo, cum_hi, lo, hi, rem)
      take = min(r_lo, gmax - len(items))
      items += [p] * take
      it += take
      cum_lo = tuple(c + max(take * l - 3.0 * (take * l) ** 0.5, 0.0) for c, l in zip(cum_lo, lo))
      cum_hi = tuple(c + take * h + 3.0 * (take * h) ** 0.5 + 1.0 for c, h in zip(cum_hi, hi))
      if take < r_lo:
        return items, (p, it, cum_lo, cum_hi)          # group full, the point surely goes on
      if r_lo != r_hi:
        return items, None                             # it may stop here or later: wait for the counters
      chain_lo, chain_hi = tuple(v * self.damp for v in lo), hi
      p, it, cum_lo, cum_hi = p + 1, 0, (0.0, 0.0), (0.0, 0.0)
    return items, ("done" if p >= self.P else (p, it, cum_lo, cum_hi))


def sim_ber_device(model, ebno_dbs, batch_size, max_mc_iter, target_bit_errs=None, target_block_errs=None,
                   early_stop=True, verbose=True, return_counters=False, lookahead=True, stats=None, profile=False,
                   group_mb=4096):
  """SURVEY 8(f) row N1: the Monte-Carlo loop of sim.py:79-133 with every step on the device, the stop rules included.

  Work item = one iteration of one SNR point: front-end kernel (bits -> encoder -> QPSK -> AWGN -> logits;
  `model.device_frontend`) into a slice of the group's buffers.  A GROUP of up to 32 items (`SweepPlanner`: further
  iterations of the point, then the first iterations of the following points where the current one is certain to stop)
  shares ONE decoder launch (bit-packed decisions), then per item a packed error count, [sharded: ONE NCCL all-reduce
  of the group's n_items x 4 int64 counters] and `polar_mc_control_group`, a one-thread kernel that walks the items in
  order through the stop rules (target bit errors, target block errors, max iterations, early stop at an error-free
  point) and ignores every item the sequential loop would not have run at that position.  Item number q of the sweep
  always draws the random numbers of offset q x batch, so ignored items hand theirs to whatever runs there next and
  the result is identical to the host loop (`sim_ber(..., on_device=False)`) for the same seed, however the items
  were grouped.  Why groups: split over 8 ranks a batch of 2^16 codewords leaves 8192 per rank = 3.46 waves of the
  list decoder's persistent grid (6.98x at 8 GPUs from the decoder alone); four such items per launch fill it.
  All buffers are allocated once per call (`group_mb` MiB of logits per group, two groups); the host reads a group's
  outcome (the sweep cursor and the per-point counters) from pinned memory while the next group is already queued.
  `lookahead=False`: one item per group, nothing queued ahead (queued == counted).
  Returns (ber, bler) like sim_ber; with return_counters also the int64 [P,4] counters, status and iterations.
  `stats` (dict, optional) receives {"queued": items launched, "counted": items counted, "groups": decoder launches};
  with `profile` also "split_us": mean device time per ITEM of front end / decoder / counter / all-reduce / control
  (CUDA events on the launching stream at the stage boundaries of each group) and the host wall time per item."""
  dist = _dist()
  rank0 = dist is None or dist.get_rank() == 0
  verbose = verbose and rank0
  dev = dk.cuda_device(model.device)
  dec = model.decoder
  if callable(getattr(model, "loop_geometry", None)):
    # decoder-domain geometry from the link model: a rate-matched code sends E channel bits of a mother code of length
    # n_polar and counts only its payload bits
    tables, n_ch, count_mask, k_count = model.loop_geometry(dev)
  else:
    frozen_pos = getattr(model.encoder, "frozen_pos", None)
    if frozen_pos is None:
      frozen_pos = dec.frozen_pos
    tables = dk.code_tables(frozen_pos, model.n, dev)
    n_ch, count_mask, k_count = model.n, tables.info_mask, tables.k
  if model._seed is None:
    model._seed = int(tc.randint(0, 2 ** 62, (1,)).item())
  ebno_dbs = np.asarray(ebno_dbs, dtype=np.float32)
  P = ebno_dbs.shape[0]
  B = int(batch_size)
  max_mc_iter = int(max_mc_iter)
  counters = np.zeros((P, 4), dtype=np.int64)
  status = np.zeros(P, dtype=np.int64)
  iters = np.zeros(P, dtype=np.int64)
  runtime = np.zeros(P)
  status_levels = ["not simulated", "reached max iter       ", "no errors - early stop",
                   "reached target bit errors", "reached target block errors"]
  fmt = "{: >9} |{: >11} |{: >11} |{: >12} |{: >12} |{: >13} |{: >12} |{: >12} |{: >10}"
  world = dist.get_world_size() if dist is not None else 1
  DEPTH = 2 if lookahead else 1
  gmax = 1
  if lookahead:
    gmax = int(max(1, min(dk.MC_GROUP_MAX, (int(group_mb) << 20) // max(B * n_ch * 4, 1), P * max_mc_iter)))
  planner = SweepPlanner(P, target_bit_errs, target_block_errs, max_mc_iter,
                         per_iter_max=(0.5 * B * k_count * world, 1.0 * B * world))
  if P == 0:
    z = tc.zeros(0, dtype=tc.float32)
    return (z, z, counters, status, iters) if return_counters else (z, z)
  offset_start = model._offset
  n_items = n_groups = 0
  marks = []                                                 # profile: (n_items, 6 timing events) per group
  with tc.cuda.device(dev):
    nw = dk.words(tables.n)
    state = tc.zeros((P, 8), dtype=tc.int64, device=dev)
    sweep = tc.zeros(8, dtype=tc.int64, device=dev)
    sizes = tc.tensor([0, 0, B * k_count, B], dtype=tc.int64, device=dev)
    slots = []
    for _ in range(DEPTH):
      slots.append(dict(u_tx=tc.empty((gmax * B, nw), dtype=tc.int32, device=dev),
                        llr=tc.empty((gmax * B, n_ch), dtype=tc.float32, device=dev),
                        u_hat=tc.empty((gmax * B, nw), dtype=tc.int32, device=dev),
                        delta=tc.zeros((gmax, 4), dtype=tc.int64, device=dev),
                        host=tc.zeros((P + 1, 8), dtype=tc.int64).pin_memory(), event=tc.cuda.Event()))

    def mark(row):
      if profile:
        e = tc.cuda.Event(enable_timing=True)
        e.record()
        row.append(e)

    def queue(slot, items, q0):
      G = len(items)
      row = []
      mark(row)
      for j, p in enumerate(items):
        model.device_frontend(tables, B, ebno_dbs[p], model._seed, offset_start + (q0 + j) * B,
                              (slot["u_tx"][j * B:(j + 1) * B], slot["llr"][j * B:(j + 1) * B]))
      mark(row)
      dec.decode_packed(slot["llr"][:G * B], tables, out=slot["u_hat"][:G * B])
      mark(row)
      delta = slot["delta"][:G]
      delta.copy_(sizes.expand(G, 4))                        # (0, 0, bits, blocks) of this rank's shard, per item
      for j in range(G):
        dk.count_errors_packed(slot["u_tx"][j * B:(j + 1) * B], slot["u_hat"][j * B:(j + 1) * B], count_mask,
                               tables.n, delta[j])
      mark(row)
      if dist is not None:
        dist.all_reduce(delta)                               # stream-ordered NCCL all-reduce of G x 4 int64
      mark(row)
      dk.mc_control_group(delta, items, state, sweep, q0, target_bit_errs, target_block_errs, max_mc_iter, early_stop)
      slot["host"][:P].copy_(state, non_blocking=True)
      slot["host"][P].copy_(sweep, non_blocking=True)
      slot["event"].record()
      mark(row)
      if profile:
        marks.append((G, row))

    known = (0, 0, (0.0, 0.0), (0.0, 0.0))                   # what the counters read back so far say
    q_known = 0
    pred, q_pred = known, 0                                  # state the queued groups lead to, if the plan holds
    inflight = []
    reported = 0                                             # points whose result line has been printed / timed
    t_point = time.perf_counter()
    nslot = 0
    finished = False
    while not finished:
      if pred is not None and pred != "done" and len(inflight) < DEPTH:
        items, after = planner.plan(pred, gmax)
        slot = slots[nslot % DEPTH]; nslot += 1
        queue(slot, items, q_pred)
        n_items += len(items); n_groups += 1
        inflight.append((slot, items, after, q_pred))
        pred, q_pred = after, q_pred + len(items)
        continue
      if not inflight:
        break
      slot, items, after, q0 = inflight.pop(0)
      slot["event"].synchronize()
      h = slot["host"].numpy()
      pc, ended, q_known = int(h[P, 0]), bool(h[P, 1]), int(h[P, 2])
      while reported < min(pc + (1 if ended and pc < P else 0), P):      # points that finished since the last look
        st = h[reported]
        counters[reported] = st[:4]; status[reported] = st[5]; iters[reported] = st[6]
        planner.finished_point(int(st[6]), int(st[0]), int(st[1]))
        now = time.perf_counter()
        runtime[reported] = now - t_point; t_point = now
        if verbose:
          i = reported
          if i == 0:
            print(fmt.format("EbNo [dB]", "BER", "BLER", "bit errors", "num bits", "block errors", "num blocks",
                             "runtime [s]", "status")); print('-' * 135)
          ber_i = counters[i, 0] / counters[i, 2] if counters[i, 2] else 0.0
          bler_i = counters[i, 1] / counters[i, 3] if counters[i, 3] else 0.0
          print(fmt.format(str(np.round(ebno_dbs[i], 3)), f"{ber_i:.4e}", f"{bler_i:.4e}", int(counters[i, 0]),
                           int(counters[i, 2]), int(counters[i, 1]), int(counters[i, 3]), np.round(runtime[i], 1),
                           status_levels[int(status[i])]))
          if status[i] == 2:
            print(f"\nSimu stopped as no error occurred @ EbNo = {ebno_dbs[i]:.1f} dB.\n")
        reported += 1
      if ended or pc >= P:
        finished = True
        break
      cum = (float(h[pc, 0]), float(h[pc, 1]))
      known = (pc, int(h[pc, 6]), cum, cum)
      as_planned = q_known == q0 + len(items) and (after is None or (after != "done" and after[0] == pc and after[1] == known[1]))
      if not as_planned:
        inflight.clear()                                     # whatever is queued behind was planned on a wrong premise:
        pred, q_pred = known, q_known                        # the control kernel ignores it; plan again from the counters
      elif not inflight:
        pred, q_pred = known, q_known                        # nothing queued ahead: plan from the exact counters
    tc.cuda.current_stream(dev).synchronize()
    model._offset = offset_start + q_known * B               # random numbers of ignored items are used again
  if stats is not None:
    stats.update(queued=int(n_items), counted=int(iters.sum()), blocks=int(counters[:, 3].sum()), groups=int(n_groups))
    if profile and marks:
      tc.cuda.synchronize(dev)
      names = ("front_end", "decode", "count", "all_reduce", "control")
      tot = float(sum(g for g, _ in marks))
      split = {nm: float(sum(r[j].elapsed_time(r[j + 1]) for _, r in marks)) / tot * 1e3 for j, nm in enumerate(names)}
      split["device_total"] = float(sum(r[0].elapsed_time(r[5]) for _, r in marks)) / tot * 1e3
      split["host_wall"] = float(runtime.sum()) / tot * 1e6
      stats["split_us"] = split
  with np.errstate(divide='ignore', invalid='ignore'):
    ber = np.nan_to_num(counters[:, 0] / counters[:, 2])
    bler = np.nan_to_num(counters[:, 1] / counters[:, 3])
  out = (tc.from_numpy(ber.astype(np.float32)), tc.from_numpy(bler.astype(np.float32)))
  if return_counters:
    return out + (counters, status, iters)
  return out


def sim_ber(mc_fun, ebno_dbs, batch_size, max_mc_iter, soft_estimates=False, target_bit_errs=None,
            target_block_errs=None, early_stop=True, verbose=True, dtype=tc.complex64, device='cpu', count_fn=None,
            on_device=True):
  """Returns (ber, bler) per SNR point; same stop rules and status codes as sim.py:19-140.
  `count_fn(b, b_hat) -> (bit_errors, block_errors)` defaults to the CUDA counter kernel; it exists so the
  sharding / stop logic can be exercised with a test double on machines without a GPU."""
  if on_device and _device_loop_ok(mc_fun, soft_estimates, count_fn):
    return sim_ber_device(mc_fun, ebno_dbs, batch_size, max_mc_iter, target_bit_errs=target_bit_errs,
                          target_block_errs=target_block_errs, early_stop=early_stop, verbose=verbose)
  count_fn = count_fn or _count
  dist = _dist()
  rank0 = dist is None or dist.get_rank() == 0
  verbose = verbose and rank0
  header = ["EbNo [dB]", "BER", "BLER", "bit errors", "num bits", "block errors", "num blocks", "runtime [s]", "status"]
  status_levels = ["not simulated", "reached max iter       ", "no errors - early stop",
                   "reached target bit errors", "reached target block errors"]
  fmt = "{: >9} |{: >11} |{: >11} |{: >12} |{: >12} |{: >13} |{: >12} |{: >12} |{: >10}"
  ebno_dbs = np.asarray(ebno_dbs, dtype=np.float32)
  num_points = ebno_dbs.shape[0]
  bit_errors = np.zeros(num_points, dtype=np.int64); block_errors = np.zeros(num_points, dtype=np.int64)
  nb_bits = np.zeros(num_points, dtype=np.int64); nb_blocks = np.zeros(num_points, dtype=np.int64)
  status = np.zeros(num_points, dtype=np.int64)
  runtime = np.zeros(num_points)

  def row(i, it, rt):
    ber = bit_errors[i] / nb_bits[i] if nb_bits[i] else 0.0
    bler = block_errors[i] / nb_blocks[i] if nb_blocks[i] else 0.0
    st = f"iter: {it:.0f}/{max_mc_iter:.0f}" if status[i] == 0 else status_levels[int(status[i])]
    return [str(np.round(ebno_dbs[i], 3)), f"{ber:.4e}", f"{bler:.4e}", int(bit_errors[i]), int(nb_bits[i]),
            int(block_errors[i]), int(nb_blocks[i]), np.round(rt, 1), st]

  for i in range(num_points):
    t0 = time.perf_counter()
    it = -1
    for ii in range(max_mc_iter):
      it += 1
      b, b_hat = mc_fun(batch_size=batch_size, ebno_db=ebno_dbs[i])[:2]
      if soft_estimates:
        b_hat = hard_decisions(b_hat)
      bit_e, block_e = count_fn(b, b_hat)
      bit_n = b.numel()
      block_n = int(b.numel() / b.shape[-1])
      if dist is not None:                       # 4 x int64 all-reduce: identical stop decisions on all ranks
        t = tc.tensor([bit_e, block_e, bit_n, block_n], dtype=tc.int64, device=b.device if b.is_cuda else 'cpu')
        dist.all_reduce(t)
        bit_e, block_e, bit_n, block_n = (int(v) for v in t.cpu())
      bit_errors[i] += bit_e; block_errors[i] += block_e
      nb_bits[i] += bit_n; nb_blocks[i] += block_n
      if verbose:
        if i == 0 and it == 0:
          print(fmt.format(*header)); print('-' * 135)
        print(fmt.format(*row(i, ii, time.perf_counter() - t0)), end="\r")
      if target_bit_errs is not None and bit_errors[i] >= target_bit_errs:
        status[i] = 3; break
      if target_block_errs is not None and block_errors[i] >= target_block_errs:
        status[i] = 4; break
      if it == max_mc_iter - 1:
        status[i] = 1
    runtime[i] = time.perf_counter() - t0
    if verbose:
      print(fmt.format(*row(i, it, runtime[i])))
    if early_stop and block_errors[i] == 0:
      status[i] = 2
      if verbose:
        print(f"\nSimu stopped as no error occurred @ EbNo = {ebno_dbs[i]:.1f} dB.\n")
      break
  with np.errstate(divide='ignore', invalid='ignore'):
    ber = np.nan_to_num(bit_errors / nb_bits)        # nan (never simulated) -> 0 (sim.py:134-139)
    bler = np.nan_to_num(block_errors / nb_blocks)
  return tc.from_numpy(ber.astype(np.float32)), tc.from_numpy(bler.astype(np.float32))
