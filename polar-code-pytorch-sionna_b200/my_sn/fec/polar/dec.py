"""my_sn decoders (my_sn/fec/polar/dec.py): the CRC-aided SCL decoder (dec.py:158-537, selection logic :507-527) --
on the min-sum list kernel it is the composed oracle of SURVEY 8(c) for BASELINE config 3 -- and the Sionna-style boxplus
SC / SCL decoders (dec.py:13-157 / :158-537, SURVEY 8f row N2).  `use_fast_scl=True` (the default) runs the list kernel
with the reference's rate-0 / REP node shortcuts (dec.py:269-306, 354-376: node-level path-metric updates, the subtree
is not descended into).  `use_hybrid_sc=True` (dec.py:437-470) decodes every codeword with SC first and list-decodes only
those whose SC decision fails the CRC (`polar_scl_decode_hybrid`: SC, a CRC check / compaction kernel and the list kernel
over the failing rows, all on the device)."""
import numpy as np
import torch as tc
from torch import nn

import d_kernels as dk
from my_sn.fec.crc import CRCEncoder, CRCDecoder


class SC_Dec(nn.Module):
  """Sionna-style SC decoder (my_sn/fec/polar/dec.py:13-157): same tree walk and leaf rule as the x_run SC_Dec,
  but the check-node update is the exact boxplus ln(1+e^(x+y)) - ln(e^x+e^y) on inputs clipped to +-30 (dec.py:33-46).
  Runs `polar_sc_decode_boxplus_f32` (the SC kernels compiled a second time with that f, csrc/polar_bp_wrap.cu).
  Parity with the CPU reference is statistical for this decoder (SURVEY 8c "secondary oracle")."""

  def __init__(self, frozen_pos, n, output_dtype=tc.float32, device='cpu'):
    super().__init__()
    self.output_dtype = output_dtype
    self.n = n
    self.frozen_pos = frozen_pos
    self.k = self.n - len(self.frozen_pos)
    self.info_pos = np.setdiff1d(np.arange(self.n), dk.to_numpy_pos(frozen_pos))
    assert self.k == len(self.info_pos), "Internal error: invalid " "info_pos generated."
    self.llr_max = 30.
    self._frozen_ind = np.zeros(self.n)
    self._frozen_ind[dk.to_numpy_pos(frozen_pos)] = 1
    self._use_fast_sc = False
    self.device = device

  def decode_packed(self, logits, tables, out=None):
    return dk.sc_decode(logits, tables, want_info=False, want_packed=True, boxplus=True, out_packed=out)[1]

  def forward(self, inputs):
    assert inputs.shape[-1] == self.n, "Last input dim must be of len n."
    assert len(inputs.shape) > 1
    dev = inputs.device if inputs.is_cuda else dk.cuda_device(self.device)
    tables = dk.code_tables(self.frozen_pos, self.n, dev)
    u_hat, _ = dk.sc_decode(inputs, tables, want_info=True, boxplus=True)
    output_shape = list(inputs.shape)
    output_shape[-1] = self.k
    output_shape[0] = -1
    out = u_hat.reshape(output_shape).to(dtype=self.output_dtype)
    return out if inputs.is_cuda else out.to(inputs.device)



class SCL_Dec(nn.Module):
  """Sionna-style list decoder (my_sn/fec/polar/dec.py:158-537) with CRC-aided selection (:507-527).
  cn_type="boxplus" (default, the reference's arithmetic): exact boxplus f in fp64; `use_fast_scl=True` (default) takes the
  path-metric update of rate-0 / REP nodes of up to 32 leaves from the node's own LLRs and skips the subtree
  (`polar_scl_decode_boxplus_pruned`), `use_fast_scl=False` updates leaf by leaf (`polar_scl_decode_boxplus`).  Parity
  with the CPU reference is statistical for both (its exp / log are the host's; SURVEY 8c).
  cn_type="minsum": the x_run min-sum list kernel under the same CRC-aided selection -- the composed oracle of
  BASELINE config 3, bit-exact against `tests/golden/sclcrc_*`.
  use_hybrid_sc=True (needs crc_degree): SC of the same arithmetic on every codeword; a codeword whose SC decision passes
  the CRC keeps it, the others are list-decoded as above.  Not the same result as full SCL: an SC decision can pass the CRC
  by chance.  `msg_pm` is then None, and `list_decoded` (device int32 [1]) holds how many codewords the last call
  list-decoded; reading it synchronises with that call."""

  def __init__(self, frozen_pos, n, list_size=8, crc_degree=None, use_hybrid_sc=False, use_fast_scl=True,
               return_crc_status=False, output_dtype=tc.float32, device='cpu', cn_type="boxplus"):
    super().__init__()
    self.device = device
    assert cn_type in ("boxplus", "minsum"), "cn_type must be 'boxplus' or 'minsum'."
    self._boxplus = cn_type == "boxplus"
    self._pruned = bool(use_fast_scl) and self._boxplus
    if output_dtype not in (tc.float16, tc.float32, tc.float64):
      raise ValueError('output_dtype must be {tf.float16, tf.float32, tf.float64}.')
    self.output_dtype = output_dtype
    n = int(n)
    assert len(frozen_pos) <= n, "Num. of elements in frozen_pos cannot be greater than n."
    assert np.log2(n) == int(np.log2(n)), "n must be a power of 2."
    assert np.log2(list_size) == int(np.log2(list_size)), "list_size must be a power of 2."
    self._n = n
    self._frozen_pos = frozen_pos
    self._k = self._n - len(self._frozen_pos)
    self._list_size = int(list_size)
    self._info_pos = np.setdiff1d(np.arange(self._n), dk.to_numpy_pos(frozen_pos))
    self._llr_max = 30.
    assert self._k == len(self._info_pos), "Internal error: invalid info_pos generated."
    if crc_degree is not None:                                   # dec.py:221-229
      self._use_crc = True
      self._crc_decoder = CRCDecoder(CRCEncoder(crc_degree, self._k))
      self._k_crc = self._crc_decoder._encoder.crc_length
      self._crc_rows_np = self._crc_decoder._encoder.syndrome_rows(self._info_pos, self._n)
    else:
      self._use_crc = False
      self._k_crc = 0
      self._crc_rows_np = None
    assert self._k >= self._k_crc, "Value of k is too small for given CRC_degree."
    if (crc_degree is None) and return_crc_status:
      raise ValueError("Returning CRC status requires given crc_degree.")
    if (crc_degree is None) and use_hybrid_sc:
      raise ValueError("Hybrid SC decoding requires given crc_degree.")
    self._use_hybrid_sc = bool(use_hybrid_sc)
    self._hybrid_mode = (dk.HYBRID_MINSUM if not self._boxplus else
                         dk.HYBRID_BOXPLUS_PRUNED if self._pruned else dk.HYBRID_BOXPLUS)
    self._return_crc_status = return_crc_status
    self._crc_rows_on = dk.PerDevice(lambda dev: dk.to_device(self._crc_rows_np, dev))
    self.msg_pm = None
    self.list_decoded = None

  @property
  def n(self): return self._n
  @property
  def k(self): return self._k
  @property
  def k_crc(self): return self._k_crc
  @property
  def frozen_pos(self): return self._frozen_pos
  @property
  def info_pos(self): return self._info_pos
  @property
  def llr_max(self): return self._llr_max
  @property
  def list_size(self): return self._list_size

  def _rows_on(self, dev):
    return (self._crc_rows_on(dev), self._k_crc) if self._use_crc else (None, 0)

  def decode_packed(self, logits, tables, out=None):
    """Device fast path of the on-device Monte-Carlo loop: bit-packed decisions of the (CRC-)selected path."""
    if self._use_hybrid_sc:
      return self._decode_hybrid(logits, tables, want_info=False, out_packed=out)["u_packed"]
    rows, ln = self._rows_on(tables.dev)
    return dk.scl_decode(logits, tables, self._list_size, crc_rows=rows, crc_len=ln, want_info=False,
                         want_packed=True, boxplus=self._boxplus, out_packed=out, pruned=self._pruned)["u_packed"]

  def _decode_hybrid(self, logits, tables, want_info, out_packed=None):
    rows, ln = self._rows_on(tables.dev)
    if self.list_decoded is None or self.list_decoded.device != tables.dev:
      self.list_decoded = tc.zeros(1, dtype=tc.int32, device=tables.dev)
    if logits.numel() == 0:
      self.list_decoded.zero_()
    return dk.scl_decode_hybrid(logits, tables, self._list_size, rows, ln, self._hybrid_mode, want_info=want_info,
                                want_packed=not want_info, out_packed=out_packed, n_list_out=self.list_decoded)

  def forward(self, inputs):
    assert inputs.dtype == self.output_dtype, "Invalid input dtype."
    assert inputs.shape[-1] == self._n, "Last input dimension must be of length n."
    assert inputs.dim() > 1
    dev = inputs.device if inputs.is_cuda else dk.cuda_device(self.device)
    tables = dk.code_tables(self._frozen_pos, self._n, dev)
    rows, ln = self._rows_on(dev)
    if self._use_hybrid_sc:                          # device path for CPU tensors too (plain copy in and out)
      u_info, self.msg_pm = self._decode_hybrid(inputs, tables, want_info=True)["u_info"], None
    elif not inputs.is_cuda and not self._boxplus:   # CPU tensor: chunked, overlapped H2D / decode / D2H inside one call
      u_info, self.msg_pm = dk.scl_decode_host(inputs, tables, self._list_size,
                                               crc_rows_np=self._crc_rows_np if self._use_crc else None, crc_len=ln)
    else:
      res = dk.scl_decode(inputs, tables, self._list_size, crc_rows=rows, crc_len=ln, want_info=True, want_pm=True,
                          boxplus=self._boxplus, pruned=self._pruned)
      u_info, self.msg_pm = res["u_info"], res["pm"]
    output_shape = list(inputs.shape)
    output_shape[-1] = self.k
    output_shape[0] = -1
    out = u_info.reshape(output_shape).to(self.output_dtype)          # CRC bits stay in the output (dec.py:527)
    if self._return_crc_status:
      raise Exception('not implement...')                              # dec.py:534-535
    return out if inputs.is_cuda else out.to(inputs.device)


class Polar5GDecoder(nn.Module):
  """Rate recovery + polar decoding + CRC removal for codewords of `Polar5GEncoder` (my_sn/fec/polar/dec.py:539-667,
  SURVEY 8f row N3).  Channel de-interleaver, de-puncturing (logit 0), de-shortening (logit -100), repetition combining
  and the sub-block de-interleaver are folded into one index plan applied by `polar_rate_recover_f32`; the decoder is the
  my_sn `SC_Dec` (boxplus SC) or the CRC-aided `SCL_Dec`.  `dec_type="hybSCL"` runs that `SCL_Dec` with
  `use_hybrid_sc=True`: SC first, list decoding only of the codewords whose SC decision fails the CRC.
  `return_crc_status=True` works here (the reference stops in a stray breakpoint, dec.py:661).  `decode_packed` (rate
  recovery, then the inner decoder's packed path) lets `sim_ber` run a 5G link model on the on-device loop."""

  def __init__(self, enc_polar, dec_type="SC", list_size=8, return_crc_status=False, output_dtype=tc.float32):
    super().__init__()
    self._output_dtype = output_dtype
    self._n_target = enc_polar.n_target; self._k_target = enc_polar.k_target
    self._n_polar = enc_polar.n_polar; self._k_polar = enc_polar.k_polar
    self._k_crc = enc_polar.enc_crc.crc_length
    self._bil = enc_polar._channel_type == "uplink"
    self._iil = False
    self._llr_max = 100
    self._enc_polar = enc_polar; self._dec_type = dec_type
    self._init_interleavers()
    if dec_type == "SC":
      print("Warning: CRC cant be used with SC dec and. Please use SCL dec.")
      self._polar_dec = SC_Dec(enc_polar._frozen_pos, self._n_polar, device=enc_polar.device)
    elif dec_type in ("SCL", "hybSCL"):
      self._polar_dec = SCL_Dec(enc_polar._frozen_pos, self._n_polar, crc_degree=enc_polar.enc_crc.crc_degree,
                                list_size=list_size, use_hybrid_sc=dec_type == "hybSCL", device=enc_polar.device)
    else:
      raise ValueError("Unknown value for dec_type.")
    assert isinstance(return_crc_status, bool), "return_crc_status must be bool."
    self._return_crc_status = return_crc_status
    if return_crc_status:
      self._dec_crc = self._polar_dec._crc_decoder if dec_type in ("SCL", "hybSCL") else CRCDecoder(enc_polar.enc_crc)
    self._plan_on = dk.PerDevice(lambda dev: tuple(dk.to_device(a, dev) for a in self._plan))
    self._rec = dk.DeviceBuffer(tc.float32)

  def _init_interleavers(self):
    """Inverse interleaver patterns (dec.py:584-598) and the fused rate-recovery plan: for polar position j,
    out[j] = fill[j], or x[src0[j]] (+ x[src1[j]] under repetition)."""
    n, e, enc = self._n_polar, self._n_target, self._enc_polar
    self.ind_ch_int_inv = np.argsort(enc.channel_interleaver(np.arange(e)))
    self.ind_sub_int_inv = np.argsort(enc.subblock_interleaving(np.arange(n)))
    self.ind_iil_inv = None
    deint = self.ind_ch_int_inv if self._bil else np.arange(e)                 # de-interleaved position -> received position
    src0 = np.full(n, -1, dtype=np.int64); src1 = np.full(n, -1, dtype=np.int64); fill = np.zeros(n, dtype=np.float32)
    p = np.arange(n)
    if e >= n:                                                                 # repetition: first E-N positions seen twice
      src0[:] = deint[p]
      rep = p[: e - n]
      src1[rep] = deint[n + rep]
    elif self._k_polar / e <= 7 / 16:                                          # puncturing: first N-E positions erased
      src0[n - e:] = deint[p[n - e:] - (n - e)]
    else:                                                                      # shortening: last N-E positions known zeros
      src0[:e] = deint[p[:e]]
      fill[e:] = -float(self._llr_max)                                         # logits: bit 0 with certainty
    inv = self.ind_sub_int_inv
    self._plan = (src0[inv].astype(np.int32), src1[inv].astype(np.int32), fill[inv].copy())

  def rate_recover(self, inputs):
    """[B, n_target] channel logits -> [B, n_polar] decoder logits (dec.py:607-634), on the GPU."""
    dev = inputs.device if inputs.is_cuda else dk.cuda_device(self._enc_polar.device)
    return dk.rate_recover(inputs.to(device=dev, dtype=tc.float32).reshape(-1, self._n_target), *self._plan_on(dev))

  def decode_packed(self, logits, tables, out=None):
    """Device fast path of the on-device Monte-Carlo loop: channel logits [B, n_target] -> rate recovery into a
    per-device buffer (grown, never shrunk) -> the inner decoder's `decode_packed` (SC, SCL or hybrid SCL) with the
    mother code's `tables`.  Returns the bit-packed decisions [B, words(n_polar)] over all n_polar positions."""
    dev = tables.dev
    x = logits.reshape(-1, self._n_target)
    B = x.shape[0]
    buf = self._rec(dev, B * self._n_polar)[:B * self._n_polar].view(B, self._n_polar)
    rec = dk.rate_recover(x, *self._plan_on(dev), out=buf)
    return self._polar_dec.decode_packed(rec, tables, out=out)

  def forward(self, inputs):
    inputs = inputs.to(tc.float32)
    input_shape = inputs.shape
    assert len(input_shape) > 1
    llr_dec = self.rate_recover(inputs)
    u_hat_crc = self._polar_dec(llr_dec)
    if self._return_crc_status:
      u_hat, crc_status = self._dec_crc(u_hat_crc)
    else:
      u_hat = u_hat_crc[:, :-self._k_crc]
    output_shape = [*input_shape]
    output_shape[-1] = self._k_target
    output_shape[0] = -1
    u_hat = u_hat.reshape(output_shape).to(dtype=self._output_dtype)
    u_hat = u_hat if inputs.is_cuda else u_hat.to(inputs.device)
    if self._return_crc_status:
      output_shape.pop()
      crc_status = crc_status.reshape(output_shape).to(dtype=self._output_dtype)
      return u_hat, (crc_status if inputs.is_cuda else crc_status.to(inputs.device))
    return u_hat
