"""Experiment configuration (mirrors x_run_sn_polar/config.py:5-26 of the reference).
pyrallis is optional: with it the dataclass is parsed exactly like the reference, without it main.py
falls back to argparse with the same flag names."""
from dataclasses import dataclass, field
from typing import List

import torch as tc


@dataclass
class PolarConfig:
  '''
  python x_run_sn_polar/main.py --k 32 --n 64 --algos [scl] --list_size 8 --bs 1000 --mc_iter 1
  '''
  k: int = 32          # number of information bits per codeword
  n: int = 64          # codeword length
  algos: List[str] = field(default_factory=lambda: ['scl'])
  kern: str = 'F2'     # unused by main (reference config.py:14)
  verbose: bool = False
  bs: int = 3
  snr_end: float = 5
  mc_iter: int = 10
  list_size: int = 8   # scl list size
  bp_iter: int = 20    # belief-propagation iterations of the `bp` curve
  mode: str = "max"
  spec: bool = False
  seed: int = 42       # main.py:24 (module-level constant in the reference)


# The reference computes this and then forces 'cpu' (config.py:25-26).  The B200 build runs the hot
# path on the GPU; on a machine without one only host-side construction (frozen sets ...) works.
device = 'cuda' if tc.cuda.is_available() else 'cpu'
