"""my_sn PolarEncoder (my_sn/fec/polar/enc.py:8-113): same transform as the x_run encoder, without a
G argument.  The gather/xor stages of G_matrix (:85-96) are the bit-packed butterfly kernel; the
reference's per-call parity self-check H.c = 0 (:110) is available as `check_parity`."""
import numpy as np
import torch as tc

from polar.enc import PolarEncoder as _Enc
import d_kernels as dk


class PolarEncoder(_Enc):
  def __init__(self, frozen_pos, n, dtype=tc.float32, device='cpu'):
    super().__init__(frozen_pos, n, None, dtype=dtype, device=device)
    self._nb_stages = int(np.log2(self._n))

  def check_parity(self, c):
    """H.c = 0 (mod 2): re-transforming a codeword must give zeros at every frozen position."""
    dev = c.device
    tables = dk.code_tables(self._frozen_pos, self._n, dev)
    u_back = dk.encode_packed(dk.pack_bits(c), self._n)              # G is an involution
    return bool(tc.all((u_back & tables.frozen_mask) == 0))


# ---------------------------------------------------------------------------------------------------------
# SURVEY 8(f) row N3: 5G NR rate matching around the polar transform (my_sn/fec/polar/enc.py:115-392).
# Everything below the CRC and the polar transform is an index permutation; it is built once on the host with
# vectorised numpy (the reference walks Python loops) and applied on the GPU by one gather kernel.
# ---------------------------------------------------------------------------------------------------------
from my_sn.fec.crc import CRCEncoder
from my_sn.fec.polar.utils import generate_5g_ranking

# TS 38.212 Table 5.4.1.1-1: sub-block interleaver pattern P(i)
_SUBBLOCK_P = np.array([0, 1, 2, 4, 3, 5, 6, 7, 8, 16, 9, 17, 10, 18, 11, 19, 12, 20, 13, 21, 14, 22, 15, 23, 24, 25, 26, 28,
                        27, 29, 30, 31])
# TS 38.212 Table 5.3.1.1-1: interleaving pattern Pi_IL^max (K_IL^max = 164)
_PI_IL_MAX = np.array([0, 2, 4, 7, 9, 14, 19, 20, 24, 25, 26, 28, 31, 34, 42, 45, 49, 50, 51, 53, 54, 56, 58, 59, 61, 62, 65, 66,
                       67, 69, 70, 71, 72, 76, 77, 81, 82, 83, 87, 88, 89, 91, 93, 95, 98, 101, 104, 106, 108, 110, 111, 113, 115,
                       118, 119, 120, 122, 123, 126, 127, 129, 132, 134, 138, 139, 140, 1, 3, 5, 8, 10, 15, 21, 27, 29, 32, 35,
                       43, 46, 52, 55, 57, 60, 63, 68, 73, 78, 84, 90, 92, 94, 96, 99, 102, 105, 107, 109, 112, 114, 116, 121,
                       124, 128, 130, 133, 135, 141, 6, 11, 16, 22, 30, 33, 36, 44, 47, 64, 74, 79, 85, 97, 100, 103, 117, 125,
                       131, 136, 142, 12, 17, 23, 37, 48, 75, 80, 86, 137, 143, 13, 18, 38, 144, 39, 145, 40, 146, 41, 147, 148,
                       149, 150, 151, 152, 153, 154, 155, 156, 157, 158, 159, 160, 161, 162, 163])


class Polar5GEncoder(PolarEncoder):
  """CRC concatenation + polar encoding + 5G rate matching to n coded bits (uplink UCI scheme; the downlink variant
  builds its tables but `forward` raises, exactly like the reference, enc.py:374-376).  No code segmentation, the
  3 parity-check bits for 12 <= k <= 19 are not used (enc.py:128-134).  `frontend_plan()` describes the code to the fused
  5G front end of `System_AWGN_model` (payload and CRC positions, CRC generator words, the rate-matching index)."""

  def __init__(self, k, n, channel_type="uplink", verbose=False, dtype=tc.float32, device='cpu'):
    k = int(k); n = int(n)
    assert n >= k, "Invalid coderate (>1)."
    assert channel_type in ("uplink", "downlink"), "Unsupported channel_type."
    self._channel_type = channel_type
    self._k_target = k; self._n_target = n
    self._verbose = verbose
    crc_degree, n_polar, frozen_pos, idx_rm, idx_input = self._init_rate_match(k, n)
    self._ind_rate_matching = idx_rm
    self._ind_input_int = idx_input
    super().__init__(frozen_pos, n_polar, dtype=dtype, device=device)
    self._enc_crc = CRCEncoder(crc_degree, k=k, dtype=dtype)
    self._idx_on = dk.PerDevice(lambda dev: dk.to_device(self._ind_rate_matching.astype(np.int32), dev))
    self._fe_plan = None

  @property
  def enc_crc(self): return self._enc_crc
  @property
  def k_target(self): return self._k_target
  @property
  def n_target(self): return self._n_target
  @property
  def k_polar(self): return self._k
  @property
  def n_polar(self): return self._n
  @property
  def k(self): return self._k_target
  @property
  def n(self): return self._n_target

  # ---- the three interleavers of TS 38.212 (index form: y = u[pattern]) ------------------------------------------
  def subblock_interleaving(self, u):
    """Sec. 5.4.1.1: 32 sub-blocks permuted by P(i); len(u) must be a multiple of 32 (enc.py:169-189)."""
    u = np.asarray(u)
    ln = u.shape[-1]
    assert np.mod(ln, 32) == 0, "len for sub-block interleaving must be a multiple of 32."
    pos = np.arange(ln)
    blk = ln // 32
    return u[_SUBBLOCK_P[pos // blk] * blk + pos % blk]

  def channel_interleaver(self, c):
    """Sec. 5.4.1.3 triangular interleaver: written row by row into a triangle of side T, read column by column,
    NULL cells skipped (enc.py:190-216)."""
    c = np.asarray(c)
    e = c.shape[-1]
    t = 0
    while t * (t + 1) // 2 < e:
      t += 1
    rows = np.repeat(np.arange(t), np.arange(t, 0, -1))                       # row index of every triangle cell
    cols = np.concatenate([np.arange(t - r) for r in range(t)]) if t else np.zeros(0, dtype=int)
    k = np.arange(rows.shape[0])                                              # write order
    valid = k < e
    order = np.lexsort((rows[valid], cols[valid]))                            # read: by column, then by row
    return c[k[valid][order]]

  def input_interleaver(self, c):
    """Sec. 5.3.1.1 input bit interleaver (downlink), defined up to 164 bits (enc.py:217-242)."""
    c = np.asarray(c)
    ln = c.shape[-1]
    assert ln <= 164, "Input interleaver only defined for length of 164."
    keep = _PI_IL_MAX[_PI_IL_MAX >= 164 - ln] - (164 - ln)
    return c[keep]

  # ---- rate-matching plan (runs once) ---------------------------------------------------------------------------
  def _init_rate_match(self, k_target, n_target):
    """(crc polynomial, n_polar, frozen_pos, rate-matching gather index [n_target], input interleaver index | None)
    following TS 38.212 Sec. 5.3.1 / 5.4.1 as the reference does (enc.py:244-361)."""
    assert n_target >= k_target, "n must be larger or equal k."
    assert n_target >= 18, "n<18 is not supported by the 5G Polar coding scheme."
    assert k_target <= 1013, "k too large - no codeword segmentation supported at the moment."
    assert n_target <= 1088, "n too large - no codeword segmentation supported at the moment."
    if self._channel_type == "uplink":
      if 12 <= k_target <= 19:
        crc_pol, k_crc = "CRC6", 6
        print("Warning: For 12<=k<=19 additional 3 parity-check bits are defined in 38.212. we didn't implement that")
      elif k_target >= 20:
        crc_pol, k_crc = "CRC11", 11
      else:
        raise ValueError("k_target<12 is not supported in 5G NR for uplink; please use 'channel coding of small block "
                         "len' scheme from Sec. 5.3.3 in 3GPP 38.212 instead.")
    else:
      assert k_target <= 140, "k too large for downlink channel config."
      assert n_target >= 25, "n too small for downlink channel config with 24 bit CRC."
      assert n_target <= 576, "n too large for downlink channel configuration."
      crc_pol, k_crc = "CRC24C", 24
    k_polar = k_target + k_crc                                                # CRC bits are information bits of the polar code
    assert k_polar <= n_target, "Device is not expected to be configured with k_polar + k_crc + n_pc > n_target."
    # mother code length, Sec. 5.3.1
    cl = np.ceil(np.log2(n_target))
    n1 = cl - 1 if (n_target <= (9 / 8) * 2 ** (cl - 1) and k_polar / n_target < 9 / 16) else cl
    n2 = np.ceil(np.log2(8 * k_polar))
    n_polar = int(2 ** max(min(n1, n2, 10), 5))
    punct = k_polar / n_target <= 7 / 16
    # pre-frozen positions, Sec. 5.4.1.1
    prefrozen = np.zeros(0, dtype=int)
    if n_target < n_polar:
      if punct:
        u = n_polar - n_target
        pat = self.subblock_interleaving(np.arange(32 * int(np.ceil(u / 32))))
        if n_target >= 3 * n_polar / 4:
          t = int(np.ceil(3 / 4 * n_polar - n_target / 2) - 1)
        else:
          t = int(np.ceil(9 / 16 * n_polar - n_target / 4) - 1)
        prefrozen = np.concatenate([pat[:u], np.arange(max(t, 0))])
      else:
        pat = self.subblock_interleaving(np.arange(n_polar))
        prefrozen = pat[n_target:n_polar]
      if self._verbose:
        print("Using %s for rate-matching." % ("puncturing" if punct else "shortening"))
    prefrozen = np.unique(prefrozen).astype(int)
    ranking, _ = generate_5g_ranking(0, n_polar, sort=False)                  # ascending reliability
    cand = ranking[~np.isin(ranking, prefrozen)]
    info_pos = np.sort(cand[-k_polar:]).astype(int)
    frozen_pos = np.setdiff1d(np.arange(n_polar), info_pos, assume_unique=True)
    ind_input = self.input_interleaver(np.arange(k_polar)) if self._channel_type == "downlink" else None
    # sub-block interleaver, circular buffer (Sec. 5.4.1.2), channel interleaver (uplink) as ONE gather index
    sub = self.subblock_interleaving(np.arange(n_polar))
    e = np.arange(n_target)
    if n_target >= n_polar:
      sel = e % n_polar                                                       # repetition
      if self._verbose: print("Using repetition coding for rate-matching")
    elif punct:
      sel = e + (n_polar - n_target)
    else:
      sel = e
    if self._channel_type == "uplink":
      sel = sel[self.channel_interleaver(e)]
    idx = sub[sel].astype(int)
    if self._verbose:
      print(f"Code params after rate-matching: k = {k_target}, n = {n_target}")
      print(f"Polar mother code: k_polar = {k_polar}, n_polar = {n_polar}")
      print("Using", crc_pol); print("Frozen positions: ", frozen_pos); print("Channel type: " + self._channel_type)
    return crc_pol, n_polar, frozen_pos, idx, ind_input

  def frontend_plan(self, dev=None):
    """The code as the fused 5G front end (`polar_nr5g_awgn_frontend`) sees it, built from this encoder's own tables:
    the payload occupies info_pos[:k] and the CRC parity bits info_pos[k:] (CRC attach + channel allocation of
    `forward`), and channel position i sends polar position `_ind_rate_matching[i]`.  Returns the host plan
    (`d_kernels.NR5GPlan`, numpy), or with `dev` its device copy (built once per device).  Downlink raises like
    `forward` does."""
    if self._channel_type == "downlink":
      raise Exception('error...')                                            # enc.py:374-376
    plan = self._fe_plan
    if plan is None:
      k, info = self._k_target, np.asarray(self.info_pos)
      plan = self._fe_plan = dk.NR5GPlan(self._n, self._n_target, info[:k],
                                         self._enc_crc.syndrome_rows(info[:k], self._n), info[k:],
                                         self._ind_rate_matching)
    return plan if dev is None else plan.on(dev)

  def forward(self, u):
    """info bits [...,k] -> rate-matched codewords [...,n] (enc.py:363-392)."""
    assert u.shape[-1] == self.k, "Last dim must be len k."
    u_crc = self._enc_crc(u)
    if self._channel_type == "downlink":
      raise Exception('error...')                                            # enc.py:374-376
    c = super().forward(u_crc)                                               # channel allocation + polar transform (GPU)
    out = dk.gather_cols(c, self._idx_on(c.device))                          # sub-block + circular buffer + channel interleaver
    shape = list(u.shape[:-1]) + [self._n_target]
    shape[0] = -1
    return out.reshape(shape).to(self.dtype)
