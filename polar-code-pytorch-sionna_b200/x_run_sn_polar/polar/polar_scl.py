"""SCL decoder with the reference call surface (x_run_sn_polar/polar/polar_scl.py:5-234).
The NumPy recursion with 2L decoder slots and a full-tree copy per information bit is replaced by one
launch of the sm_100a kernel `polar_scl_decode` (csrc/polar_scl_api.cu): fp64 tree and path metrics,
lazy copy-on-write through per-stage pointer tables, warp bitonic ranking of the 2L candidates."""
import numpy as np
import torch as tc
from torch import nn

import d_kernels as dk


class SCL_Dec(nn.Module):
  def __init__(self, frozen_pos, n, list_size=8, crc_degree=None, use_hybrid_sc=False, use_fast_scl=True,
               return_crc_status=False, output_dtype=tc.float32, device='cpu'):
    super().__init__()
    self.device = device
    if output_dtype not in (tc.float16, tc.float32, tc.float64):
      raise ValueError('output_dtype must be {tf.float16, tf.float32, tf.float64}.')
    self.output_dtype = output_dtype
    n = int(n)
    assert len(frozen_pos) <= n, "Num. of elements in frozen_pos cannot be greater than n."
    assert np.log2(n) == int(np.log2(n)), "n must be a power of 2."
    assert np.log2(list_size) == int(np.log2(list_size)), "list_size must be a power of 2."
    assert list_size <= dk.SCL_MAX_L, "list_size must be <= %d." % dk.SCL_MAX_L
    self._n = n
    self._frozen_pos = frozen_pos
    self._k = self._n - len(self._frozen_pos)
    self._list_size = int(list_size)
    self._info_pos = np.setdiff1d(np.arange(self._n), dk.to_numpy_pos(frozen_pos))
    self._llr_max = 30.
    assert self._k == len(self._info_pos), "Internal error: invalid info_pos generated."
    self._n_stages = int(np.log2(self._n))
    # crc_degree / use_hybrid_sc / use_fast_scl / return_crc_status are accepted and ignored, exactly
    # like the reference (polar_scl.py:16-19); the CRC-aided decoder is my_sn.fec.polar.dec.SCL_Dec.
    self.msg_pm = None

  @property
  def n(self): return self._n
  @property
  def k(self): return self._k
  @property
  def frozen_pos(self): return self._frozen_pos
  @property
  def info_pos(self): return self._info_pos
  @property
  def list_size(self): return self._list_size
  @property
  def llr_max(self): return self._llr_max

  def decode_packed(self, logits, tables, out=None):
    """Device fast path of the on-device Monte-Carlo loop: bit-packed decisions of the best path."""
    return dk.scl_decode(logits, tables, self._list_size, want_info=False, want_packed=True, out_packed=out)["u_packed"]

  def forward(self, inputs):
    assert inputs.dtype == self.output_dtype, "Invalid input dtype."
    assert inputs.shape[-1] == self._n, "Last input dim must be of len n."
    assert inputs.dim() > 1
    dev = inputs.device if inputs.is_cuda else dk.cuda_device(self.device)
    tables = dk.code_tables(self._frozen_pos, self._n, dev)
    if inputs.is_cuda:
      res = dk.scl_decode(inputs, tables, self._list_size, want_info=True, want_pm=True)
      u_info, self.msg_pm = res["u_info"], res["pm"]   # [B, L] ascending (reference keeps [B, 2L] duplicates)
    else:         # CPU tensor in -> CPU tensor out (the reference's boundary): chunked, overlapped H2D / decode / D2H
      u_info, self.msg_pm = dk.scl_decode_host(inputs, tables, self._list_size)
    output_shape = list(inputs.shape)
    output_shape[-1] = self.k
    output_shape[0] = -1
    return u_info.reshape(output_shape).to(self.output_dtype)
