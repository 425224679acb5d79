"""Ordered-statistics decoder (my_sn/fec/osd/dec.py:8-192) on the GPU: `polar_osd_decode` (csrc/polar_osd.cu) does the
whole decode of a codeword -- reliability sort, most-reliable basis, error-pattern search -- in one CTA.  Same
constructor, attributes, error behaviour and output (all n codeword bits, fp) as the reference's OSDecoder."""
import math

import numpy as np
import torch as tc
from torch import nn

import d_kernels as dk


class OSDecoder(nn.Module):
  def __init__(self, t=0, encoder=None, dtype=tc.float32, device='cpu'):
    super().__init__()
    self.device = device
    self.dtype = dtype
    self._llr_max = 100.                      # internal clipping value (dec.py:30)
    if dtype not in (tc.float16, tc.float32, tc.float64):
      raise ValueError('dtype must be {tf.float16, tf.float32, tf.float64}.')
    assert (int(t) == t), "t must be int."
    self._t = int(t)
    if encoder.k is None:
      raise AttributeError("It seems as if encoder is not init or has no attribute k.")
    # generator matrix: the encoder applied to the k unit vectors (dec.py:40-42)
    u = tc.eye(encoder.k, device=device)
    self._gm = encoder(u).to(dtype)
    self._k = self._gm.size(0)
    self._n = self._gm.size(1)
    num_patterns = math.comb(self._n, self._t)            # dec.py:46-53: the reference sizes its check with C(n, t)
    num_symbols = num_patterns * self._n
    if num_symbols > 1e9:
      print(f"Note: Required memory complexity is large for given code params and t={t}. Please consider small batch-sizes")
    if num_symbols > 1e11:
      raise ResourceWarning("OSD cant run this (complexity too high). Please use a smaller value for t.")
    # the error patterns themselves (dec.py:54-56) are enumerated inside the kernel, in itertools.combinations order
    self._gm_rows_np = dk.pack_rows(self._gm.detach().cpu().numpy())
    self._gm_rows_on = dk.PerDevice(lambda dev: dk.to_device(self._gm_rows_np, dev))

  @property
  def gm(self): return self._gm
  @property
  def n(self): return self._n
  @property
  def k(self): return self._k
  @property
  def t(self): return self._t

  def forward(self, inputs):
    """inputs [..., n] channel logits ln P(1)/P(0) -> [..., n] hard decisions of all codeword bits (dec.py:149-191)."""
    input_shape = inputs.shape
    dev = dk.cuda_device(inputs.device if inputs.is_cuda else None)
    x = inputs.reshape(-1, self._n).to(self.dtype)
    res = dk.osd_decode(x, self._gm_rows_on(dev), self._n, self._k, self._t)
    c_hat = res["c"].reshape(input_shape).to(self.dtype)
    return c_hat if inputs.is_cuda else c_hat.to(inputs.device)
