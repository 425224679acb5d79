"""End-to-end AWGN link model with the reference call surface (z_sys_model/awgn_model.py:16-44).

`forward(batch_size, ebno_db) -> (bits, bits_hat)`.  With `fused=True` (default) everything before the
decoder -- BinarySource, PolarEncoder, QPSK Mapper, AWGN, Demapper -- is one launch of
`polar_awgn_frontend` (Philox counter RNG, closed-form logit -2.sqrt2.y/no); with `fused=False` the
reference's layer-by-layer composition is used (same statistics, torch RNG on the model's device).

5G codes: with an encoder that has `frontend_plan` (`Polar5GEncoder`), n is the number of channel bits E and k the
payload length, as in the reference (`System_AWGN_model(E, k, Polar5GEncoder(k, E), Polar5GDecoder(enc, ...))`).  The
fused path is then one launch of `polar_nr5g_awgn_frontend` (payload, CRC, channel allocation, polar transform, rate
matching, QPSK/AWGN, demapper) and `bits` is the [B, k] payload; the code rate stays k / E.  `cw_estimates=True` is not
available there (the front end returns the payload, not the rate-matched codeword)."""
import torch as tc
from torch import nn

from my_sn.trans.channel import awgn
from my_sn.trans import mapping, binary_source, ebno
import d_kernels as dk


class System_AWGN_model(nn.Module):
  def __init__(self, n, k, encoder, decoder, cw_estimates=False, device='cpu', fused=True, seed=None):
    super().__init__()
    self.cw_estimates = cw_estimates
    self.n_bits_per_sym = 2
    self.n = n
    self.k = k
    self.coderate = self.k / self.n
    self.device = device
    self.fused = fused
    self.encoder = encoder
    self.decoder = decoder
    self._seed = seed
    self._offset = 0
    self._layers = None
    self._nr5g = callable(getattr(encoder, "frontend_plan", None))     # rate-matched 5G code: payload k, E channel bits
    if self._nr5g:
      assert n == encoder.n and k == encoder.k, "n and k must be the 5G encoder's channel bits E and payload bits k."
      if fused and cw_estimates:
        raise ValueError("cw_estimates=True is not supported by the fused 5G front end; use fused=False.")

  def _build_layers(self, dev):
    self.constell = mapping.QamConstell(self.n_bits_per_sym, device=dev)
    self.mapper = mapping.Mapper(constell=self.constell, device=dev)
    self.demapper = mapping.Demapper(constell=self.constell)
    self.binary_src = binary_source.BinarySource(device=dev)
    self.awgn_channel = awgn.AWGN(device=dev)
    self._layers = dev

  def _frozen_pos(self):
    frozen_pos = getattr(self.encoder, "frozen_pos", None)
    return self.decoder.frozen_pos if frozen_pos is None else frozen_pos

  def loop_geometry(self, dev):
    """What the on-device Monte-Carlo loop (my_sn/sim.py::sim_ber_device) needs to know about the code: (CodeTables of
    the code the decoder decodes, channel logits per codeword, device mask of the counted positions, counted bits per
    codeword).  A plain code counts its information positions; a 5G code the k payload positions of its mother code."""
    if self._nr5g:
      plan = self.encoder.frontend_plan(dev)
      return dk.code_tables(self._frozen_pos(), plan.n, dev), plan.e, plan.payload_mask_d, plan.k
    tables = dk.code_tables(self._frozen_pos(), self.n, dev)
    return tables, self.n, tables.info_mask, tables.k

  def device_frontend(self, tables, batch_size, ebno_db, seed, offset, out):
    """Hook of the on-device Monte-Carlo loop (my_sn/sim.py::sim_ber_device): one launch of polar_awgn_frontend (5G:
    polar_nr5g_awgn_frontend) into the caller-owned buffers out = (u_packed, logits).  A link model without this method
    runs the host loop."""
    no = ebno.ebnodb2no(float(ebno_db), self.n_bits_per_sym, self.coderate)
    if self._nr5g:
      dk.nr5g_awgn_frontend(self.encoder.frontend_plan(tables.dev), batch_size, no, seed, offset, out=out)
    else:
      dk.awgn_frontend(tables, batch_size, no, seed, offset, out=out)

  def forward(self, batch_size, ebno_db):
    dev = dk.cuda_device(self.device)
    no = ebno.ebnodb2no(float(ebno_db), self.n_bits_per_sym, self.coderate)
    if self.fused and self._nr5g:
      plan = self.encoder.frontend_plan(dev)
      if self._seed is None:
        self._seed = int(tc.randint(0, 2 ** 62, (1,)).item())
      u_packed, _, llr = dk.nr5g_awgn_frontend(plan, batch_size, no, self._seed, self._offset)
      self._offset += int(batch_size)
      bits_hat = self.decoder(llr)
      return dk.unpack_info(u_packed, plan.payload_pos_d, plan.n), bits_hat
    if self.fused:
      tables = dk.code_tables(self._frozen_pos(), self.n, dev)
      if self._seed is None:           # derive the Philox key from torch's seeded generator (set_seed, main.py:25-29)
        self._seed = int(tc.randint(0, 2 ** 62, (1,)).item())
      u_packed, c_packed, llr = dk.awgn_frontend(tables, batch_size, no, self._seed, self._offset,
                                                 want_codeword=self.cw_estimates)
      self._offset += int(batch_size)
      bits_hat = self.decoder(llr)
      if self.cw_estimates:
        pos = tc.arange(self.n, dtype=tc.int32, device=dev)
        return dk.unpack_info(c_packed, pos, self.n), bits_hat
      return dk.unpack_info(u_packed, tables.info_pos, self.n), bits_hat
    if self._layers != dev:
      self._build_layers(dev)
    bits = self.binary_src([batch_size, self.k])
    codewords = self.encoder(bits)
    x = self.mapper(codewords)
    y = self.awgn_channel([x, no])
    llr = self.demapper([y, no])
    bits_hat = self.decoder(llr)
    if self.cw_estimates:
      return codewords, bits_hat
    return bits, bits_hat
