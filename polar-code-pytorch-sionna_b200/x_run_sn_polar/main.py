"""CLI of the experiment (mirrors x_run_sn_polar/main.py:25-78): SC (always), SCL and belief-propagation BLER curves over
Eb/N0 = 0:0.5:snr_end for an RM-rule polar code, on the GPU.  `--algos [scl,bp]` picks the extra curves; `bp` adds
`BP-<bp_iter>` (boxplus BP, my_sn BP_Dec).

  python x_run_sn_polar/main.py --k 32 --n 64 --algos [scl] --bs 100 --mc_iter 1      (README command)
  torchrun --nproc-per-node 8 x_run_sn_polar/main.py ...   shards every batch over the ranks (bs is per rank)
"""
import math
import os
import random
import sys
from os.path import dirname

sys.path.append(dirname(dirname(os.path.abspath(__file__))))
sys.path.append(dirname(os.path.abspath(__file__)))
import numpy as np
import torch as tc

from my_sn.plotting import PlotBER
from polar.enc import PolarEncoder as PolarEnc2
from polar.polar_scl import SCL_Dec
from polar.polar_sc import SC_Dec
from my_sn.fec.polar.dec import BP_Dec
from config import PolarConfig, device
from z_sys_model.awgn_model import System_AWGN_model
from d_kernels import *  # noqa: F401,F403  F2, F4.., gen_arikan (main.py:30)
from d_kernels import F2
from polar.froze import get_Kern_frozen_bits, get_Kern_frozen_bits2  # noqa: F401


def set_seed(seed):
  np.random.seed(seed)
  random.seed(seed)
  tc.manual_seed(seed)


def gen_code(c, Gn, name, mode='sc'):
  a = math.log(c.n, 2); assert a.is_integer()
  G_, G_weights, frozen_pos = get_Kern_frozen_bits(c.n, c.n - c.k, Gn)
  enc = PolarEnc2(frozen_pos, c.n, G_, device=device)
  if mode == "sc": dec = SC_Dec(frozen_pos, c.n, device=device)
  elif mode == "scl": dec = SCL_Dec(frozen_pos, c.n, c.list_size, device=device)
  elif mode == "bp": dec = BP_Dec(frozen_pos, c.n, num_iter=c.bp_iter, device=device)
  else: raise Exception('error...')
  return [System_AWGN_model(c.n, c.k, enc, dec, device=device), name]


def parse_config(argv=None):
  try:
    import pyrallis
    return pyrallis.parse(config_class=PolarConfig, args=argv)
  except ImportError:
    import argparse
    ap = argparse.ArgumentParser()
    import typing
    d = PolarConfig()
    hints = typing.get_type_hints(PolarConfig)                     # the annotation decides (snr_end: float = 5)
    for f, v in vars(d).items():
      t = hints.get(f, type(v))
      if t is bool: ap.add_argument("--" + f, type=lambda s: s.lower() in ("1", "true", "yes"), default=v)
      elif isinstance(v, list): ap.add_argument("--" + f, type=lambda s: [t for t in s.strip("[]").split(",") if t], default=v)
      else: ap.add_argument("--" + f, type=t if t in (int, float, str) else type(v), default=v)
    return PolarConfig(**vars(ap.parse_args(argv)))


def main(c: PolarConfig):
  import torch.distributed as dist
  if "RANK" in os.environ and not dist.is_initialized():       # launched under torchrun: one rank per GPU
    tc.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dist.init_process_group("nccl")
  rank = dist.get_rank() if dist.is_initialized() else 0
  k = c.k; n = c.n
  ebno_db = np.arange(0, c.snr_end, 0.5)
  codes_under_test = [gen_code(c, F2, "SC", mode="sc")]
  if 'scl' in c.algos:
    codes_under_test.append(gen_code(c, F2, f"SCL-{c.list_size}", mode="scl"))
  if 'bp' in c.algos:
    codes_under_test.append(gen_code(c, F2, f"BP-{c.bp_iter}", mode="bp"))
  ber_plot = PlotBER(f"Performance of Short Len Codes (k={k}, n={n})")
  for code in codes_under_test:
    if rank == 0: print("\nRunning: " + code[-1])
    set_seed(c.seed + rank)                                       # main.py:57 (per-rank stream when sharded)
    ber_plot.simulate(code[0], ebno_dbs=ebno_db, batch_size=c.bs, target_block_errs=1000, legend=code[-1],
                      soft_estimates=False, max_mc_iter=c.mc_iter, add_bler=True, device=device)
  if rank == 0:
    for name, curve in zip(ber_plot.legend, ber_plot.ber):
      print("%-14s" % name, np.array2string(curve.numpy(), precision=5, separator=", "))
    try:
      import matplotlib.pyplot as plt
      plt.figure(figsize=(16, 12)); plt.title(f"SC vs scl (k={k},n={n})", fontsize=25); plt.grid(which="both")
      plt.xlabel(r"$E_b/N_0$ (dB)", fontsize=25); plt.ylabel(r"BLER", fontsize=25)
      for i, name in enumerate(ber_plot.legend):
        if "BLER" in name:
          plt.semilogy(ebno_db, ber_plot.ber[i], c='C%d' % i, label=name, linewidth=2, linestyle='--' if "SC " in name else '-')
      plt.legend(fontsize=20); plt.xlim([0, 4.5])
      os.makedirs('./x_run_sn_polar/plots', exist_ok=True)
      plt.savefig(f'./x_run_sn_polar/plots/sc_{c.mc_iter=}_{c.bs=}.png')
    except ImportError:
      pass
  return ber_plot


if __name__ == '__main__':
  main(parse_config())
