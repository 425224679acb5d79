"""d_kernels.py -- loader of the sm_100a kernel library (C ABI, include/polar_b200.h).

In the reference this module holds the *polarization kernel matrices* (x_run_sn_polar/d_kernels.py:3-11:
`gen_arikan`, `F2`, `F4`..`F32`), star-imported by main.py:30.  Those names are kept.  The B200 build
also makes it the single place where `libpolar_b200.so` is loaded (ctypes) and where torch tensors
are turned into raw device pointers: every decoder / encoder / link-model class in this package
calls the CUDA kernels through the functions below.  There is NO CPU fallback: if the library is
missing, or no CUDA device is present when a kernel is requested, these functions raise.
"""
import copy
import ctypes
import os

import numpy as np
import torch as tc

from config import device  # noqa: F401  (re-exported: main.py star-imports this module)

# ---- polarization kernels (reference d_kernels.py:3-11) -----------------------------------------


def gen_arikan(F2, lay):
  """F2^{(x) lay} (Kronecker power), reference d_kernels.py:3-7."""
  FN = tc.clone(F2)
  for _ in range(lay - 1):
    FN = tc.kron(F2, FN)
  return FN


# Host tensors: frozen-set construction (froze.py) is host-side, and creating them on `device` at import time would open a
# CUDA context on GPU 0 in every torchrun rank before main.py selects LOCAL_RANK.
F2 = tc.tensor([[1, 0], [1, 1]], dtype=tc.float32, device='cpu')
F4 = gen_arikan(F2, 2); F8 = gen_arikan(F2, 3)
F16 = gen_arikan(F2, 4); F32 = gen_arikan(F2, 5)

# ---- library loading ------------------------------------------------------------------------------
_PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("POLAR_B200_LIB", os.path.join(_PKG_DIR, "libpolar_b200.so"))
_lib = None

POLAR_OK, POLAR_EINVAL, POLAR_EALIGN, POLAR_ENOMEM, POLAR_ECUDA = 0, -1, -2, -3, -4
SC_MAX_N, SCL_MAX_N, SCL_MAX_L, BP_MAX_N = 8192, 4096, 32, 1024

_vp, _i32, _i64, _u64, _f32, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64,
                                    ctypes.c_float, ctypes.c_size_t)
_SIGNATURES = {
  # name: (restype, argtypes)   -- must match include/polar_b200.h
  "polar_last_error": (ctypes.c_char_p, []),
  "polar_version": (ctypes.c_char_p, []),
  "polar_launch_count": (ctypes.c_ulonglong, []),
  "polar_init": (_i32, [_i32]),
  "polar_set_option": (_i32, [ctypes.c_char_p, _i32]),
  "polar_clear_options": (None, []),
  "polar_sc_decode_f32": (_i32, [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _i32, _vp]),
  "polar_sc_decode_boxplus_f32": (_i32, [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _i32, _vp]),
  "polar_scl_workspace_bytes": (_sz, [_i32, _i32, _i64]),
  "polar_scl_decode": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _sz, _vp]),
  "polar_scl_boxplus_workspace_bytes": (_sz, [_i32, _i32, _i64]),
  "polar_scl_decode_boxplus": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _sz, _vp]),
  "polar_scl_decode_boxplus_pruned": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _sz, _vp]),
  "polar_scl_hybrid_workspace_bytes": (_sz, [_i32, _i32, _i64, _i32]),
  "polar_scl_decode_hybrid": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
  "polar_belief_decode_f32": (_i32, [_vp, _vp, _i32, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
  "polar_encode_packed": (_i32, [_vp, _i32, _i64, _vp, _vp]),
  "polar_encode_f32": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp]),
  "polar_gather_cols_f32": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp]),
  "polar_rate_recover_f32": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _vp]),
  "polar_awgn_frontend": (_i32, [_u64, _u64, _f32, _vp, _i32, _i64, _vp, _vp, _vp, _vp]),
  "polar_nr5g_awgn_frontend": (_i32, [_u64, _u64, _f32, _vp, _vp, _vp, _i32, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp]),
  "polar_bec_frontend": (_i32, [_u64, _u64, _f32, _f32, _vp, _i32, _i64, _vp, _vp, _vp, _vp]),
  "polar_bec_llr": (_i32, [_u64, _u64, _f32, _f32, _vp, _i32, _i64, _vp, _vp]),
  "polar_qpsk_awgn_llr": (_i32, [_u64, _u64, _f32, _vp, _i32, _i64, _vp, _vp]),
  "polar_count_errors_packed": (_i32, [_vp, _vp, _vp, _i32, _i64, _vp, _vp]),
  "polar_count_errors_f32": (_i32, [_vp, _vp, _i32, _i64, _vp, _vp]),
  "polar_mc_control_group": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong,
                                    ctypes.c_longlong, _i32, _vp]),
  "polar_osd_decode": (_i32, [_vp, _vp, _i32, _i32, _i32, _i64, _vp, _vp, _vp, _vp]),
  "polar_scl3_math_selftest": (_i32, [ctypes.c_uint64, _vp, _vp]),
  "polar_pack_bits_f32": (_i32, [_vp, _i32, _i64, _vp, _vp]),
  "polar_unpack_info_f32": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp]),
  "polar_sc_decode_host": (_i32, [_vp, _vp, _i32, _i64, _vp, _i32]),
  "polar_scl_decode_host": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _i32, _i32]),
  "polar_sc_decode_host_f32": (_i32, [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _i32, _i32]),
  "polar_scl_decode_host_f32": (_i32, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _i32]),
}


def lib():
  """The loaded C-ABI library.  Raises (never falls back) when it is missing."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise RuntimeError(
        "polar_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(there is no CPU fallback)" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
      fn = getattr(L, name)        # AttributeError if the library does not export a declared symbol
      fn.restype = res
      fn.argtypes = args
    _lib = L
  return _lib


class PolarKernelError(RuntimeError):
  pass


def check(rc):
  """Turn a POLAR_E* return code into an exception carrying polar_last_error()."""
  if rc == POLAR_OK:
    return
  msg = lib().polar_last_error().decode("utf-8", "replace")
  if rc == POLAR_EINVAL:
    raise AssertionError(msg)            # the reference signals bad shapes / sizes with assert
  if rc == POLAR_ENOMEM:
    raise MemoryError(msg)
  raise PolarKernelError("polar_b200 error %d: %s" % (rc, msg))


def cuda_device(dev=None):
  """Resolve the CUDA device kernels run on.  Fails loudly on a machine without a GPU."""
  if not tc.cuda.is_available():
    raise RuntimeError("polar_b200: no CUDA device available -- the decoders/encoder/front end run only "
                       "on the GPU (sm_100a); there is no CPU fallback")
  if dev is None or str(dev) == "cpu":
    return tc.device("cuda", tc.cuda.current_device())
  dev = tc.device(dev)
  if dev.type != "cuda":
    raise RuntimeError("polar_b200: device %s is not a CUDA device" % dev)
  if dev.index is None:
    dev = tc.device("cuda", tc.cuda.current_device())
  return dev


def ptr(t):
  return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def stream_ptr(dev):
  return ctypes.c_void_p(tc.cuda.current_stream(dev).cuda_stream)


def words(n):
  return 1 if n < 32 else n // 32


# ---- host-side code description ---------------------------------------------------------------------
def to_numpy_pos(frozen_pos):
  """frozen_pos may be a NumPy int array or a torch int64 tensor (main.py passes a tensor)."""
  if isinstance(frozen_pos, tc.Tensor):
    return frozen_pos.detach().cpu().numpy().astype(np.int64)
  return np.asarray(frozen_pos).astype(np.int64)


def pack_rows(m):
  """0/1 matrix [r, n] (numpy) -> uint32 bit-packed rows [r, (n+31)//32], position i = bit i%32 of word i//32 (as int32).
  The one bit packer of the host tables: frozen masks, 5G payload masks, OSD generator rows."""
  m = np.asarray(m) != 0
  r, n = m.shape
  bits = np.zeros((r, (n + 31) // 32 * 32), dtype=np.uint8)
  bits[:, :n] = m
  return np.packbits(bits.reshape(r, -1, 32), axis=2, bitorder="little").view(np.int32).reshape(r, -1)


def frozen_mask_words(pos, n):
  """uint32[words(n)]: bit (i % 32) of word (i // 32) set <=> position i in `pos` (the frozen set of a code, or the payload
  positions of a 5G code)."""
  row = np.zeros((1, n), dtype=np.uint8)
  row[0, to_numpy_pos(pos)] = 1
  return pack_rows(row)[0].view(np.uint32)


def to_device(a, dev):
  """Device copy of host array `a`; uint32 bit patterns are stored as int32, the type the kernel wrappers pass."""
  a = np.asarray(a)
  return tc.from_numpy((a.view(np.int32) if a.dtype == np.uint32 else a).copy()).to(dev)


def _indexed(dev):
  """`dev` as a torch.device with an explicit index (`cuda` = the current device): the key of every per-device store."""
  dev = tc.device(dev)
  return tc.device("cuda", tc.cuda.current_device()) if dev.type == "cuda" and dev.index is None else dev


class PerDevice:
  """Objects made by `build(dev, *key)` once per (device, key) and kept: device copies of host tables, or objects derived
  from them.  Each owner (a decoder, a plan, this module) holds its own."""

  def __init__(self, build):
    self._build, self._made = build, {}

  def __call__(self, dev, *key):
    k = (_indexed(dev),) + key
    obj = self._made.get(k)
    if obj is None:
      obj = self._made[k] = self._build(*k)
    return obj


class DeviceBuffer:
  """Scratch memory: one flat `dtype` buffer per device, replaced by one of `numel + slack` elements whenever a call needs
  more than it holds, never shrunk.  All streams of a device share it, so two streams must not use it at the same time."""

  def __init__(self, dtype, slack=0):
    self._dtype, self._slack, self._bufs = dtype, slack, {}

  def __call__(self, dev, numel):
    dev = _indexed(dev)
    buf = self._bufs.get(dev)
    if buf is None or buf.numel() < numel:
      buf = self._bufs[dev] = tc.empty(numel + self._slack, dtype=self._dtype, device=dev)
    return buf


_INITIALISED = set()


def init_device(dev):
  """polar_init(device) once per device: the only call of the library that allocates on its own (SC stage scratch)."""
  idx = dev.index if dev.index is not None else tc.cuda.current_device()
  if idx not in _INITIALISED:
    check(lib().polar_init(int(idx)))
    _INITIALISED.add(idx)
  return idx


def set_option(name, value):
  """Tuning / test override of a POLAR_* option (include/polar_b200.h: polar_set_option)."""
  check(lib().polar_set_option(name.encode(), int(value)))


def clear_options():
  lib().polar_clear_options()


class CodeTables:
  """Device-resident description of one (frozen set, n) code, shared by encoder/decoders/front end."""

  def __init__(self, frozen_pos, n, dev):
    self.n = int(n)
    self.dev = dev
    init_device(dev)
    fp = to_numpy_pos(frozen_pos)
    self.info_pos_np = np.setdiff1d(np.arange(self.n), fp)          # ascending (polar_sc.py:19)
    self.k = int(self.info_pos_np.shape[0])
    self.mask_np = frozen_mask_words(fp, self.n)
    rank = np.full(self.n, -1, dtype=np.int32)
    rank[self.info_pos_np] = np.arange(self.k, dtype=np.int32)
    self.frozen_mask = to_device(self.mask_np, dev)
    self.info_pos = to_device(self.info_pos_np.astype(np.int32), dev)
    self.info_rank = to_device(rank, dev)
    self.info_mask = to_device((~self.mask_np) & (np.uint32(0xFFFFFFFF) if self.n >= 32 else np.uint32((1 << self.n) - 1)), dev)


class NR5GPlan:
  """What polar_nr5g_awgn_frontend needs to know about one rate-matched 5G code (Polar5GEncoder.frontend_plan).
  Host fields (numpy): n (mother code), e (channel bits), k (payload bits), crc_len, payload_pos [k], payload_mask
  [words(n)] uint32, crc_rows [n] uint32, crc_pos [crc_len], rm_idx [e].  `on(dev)` returns the plan with the device
  copies payload_mask_d / crc_rows_d / crc_pos_d / rm_idx_d / payload_pos_d (int32), built once per device; `dev` is
  None on the host plan."""

  def __init__(self, n, e, payload_pos, crc_rows, crc_pos, rm_idx):
    self.n, self.e = int(n), int(e)
    self.payload_pos = np.asarray(payload_pos, dtype=np.int64)
    self.k = int(self.payload_pos.shape[0])
    self.crc_rows = np.asarray(crc_rows, dtype=np.uint32)
    self.crc_pos = np.asarray(crc_pos, dtype=np.int64)
    self.crc_len = int(self.crc_pos.shape[0])
    self.rm_idx = np.asarray(rm_idx, dtype=np.int64)
    self.payload_mask = frozen_mask_words(self.payload_pos, self.n)
    self.dev = None
    self._on = PerDevice(self._device_copy)

  def on(self, dev):
    return self._on(dev)

  def _device_copy(self, dev):
    init_device(dev)
    p = copy.copy(self)
    p.dev = dev
    p.payload_mask_d, p.crc_rows_d = to_device(self.payload_mask, dev), to_device(self.crc_rows, dev)
    p.crc_pos_d, p.rm_idx_d, p.payload_pos_d = (to_device(a.astype(np.int32), dev)
                                                for a in (self.crc_pos, self.rm_idx, self.payload_pos))
    return p


_code_tables = PerDevice(lambda dev, fp, n: CodeTables(np.frombuffer(fp, dtype=np.int64), n, dev))


def code_tables(frozen_pos, n, dev):
  """The CodeTables of (frozen set, n) on `dev`, built on first use."""
  return _code_tables(dev, to_numpy_pos(frozen_pos).tobytes(), int(n))


# ---- kernel wrappers (device tensors in, device tensors out) -------------------------------------------
_workspace = DeviceBuffer(tc.uint8, slack=256)      # the list decoders' workspace


def _call(dev, name, *args, workspace=None):
  """Run library function `name` on `dev` with `args` and the device's current stream; raise on its error code.
  workspace = (size function name, its args): the list-decoder workspace (NULL when 0 bytes) and its size go before the
  stream.  The size is asked on `dev`: it depends on the device's SM count."""
  with tc.cuda.device(dev):
    if workspace is not None:
      need = int(getattr(lib(), workspace[0])(*workspace[1]))
      args += (ptr(_workspace(dev, need)) if need else None, need)
    check(getattr(lib(), name)(*args, stream_ptr(dev)))


def _out(dev, shape, dtype, want=True, given=None):
  """An output of a wrapper: the caller-owned buffer `given` if any, else a new tensor if the output is wanted, else None."""
  if given is not None:
    return given
  return tc.empty(shape, dtype=dtype, device=dev) if want else None


def _philox_key(seed):
  return int(seed) & 0xFFFFFFFFFFFFFFFF


def _stop_target(target):
  return -1 if target is None else int(target)     # -1: the rule is disabled


def _prep_logits(x, n, dev):
  x = x.to(device=dev, dtype=tc.float32).reshape(-1, n)
  if not x.is_contiguous() or x.data_ptr() % 16:
    x = x.contiguous().clone() if x.data_ptr() % 16 else x.contiguous()
  return x


def _rows(x):
  return x.to(tc.float32).reshape(-1, x.shape[-1]).contiguous()


def sc_decode(logits, tables, want_info=True, want_packed=False, boxplus=False, out_packed=None):
  """polar_sc_decode_f32 (min-sum f) or polar_sc_decode_boxplus_f32 (exact boxplus f, my_sn SC_Dec).
  logits [B,n] (any float dtype/device) -> (u_info fp32 [B,k] | None, u_packed int32 | None).
  out_packed: caller-owned int32 [B, words(n)] buffer for the packed decisions (Monte-Carlo loop: no allocation per call)."""
  dev = tables.dev
  x = _prep_logits(logits, tables.n, dev)
  B = x.shape[0]
  u_info = _out(dev, (B, tables.k), tc.float32, want_info)
  u_packed = _out(dev, (B, words(tables.n)), tc.int32, want_packed, out_packed)
  _call(dev, "polar_sc_decode_boxplus_f32" if boxplus else "polar_sc_decode_f32", ptr(x), ptr(tables.frozen_mask), tables.n,
        B, ptr(u_packed), ptr(u_info), ptr(tables.info_pos), tables.k)
  return u_info, u_packed


def scl_decode(logits, tables, list_size, crc_rows=None, crc_len=0, want_info=True, want_packed=False,
               want_pm=False, want_list=False, boxplus=False, out_packed=None, pruned=False):
  """polar_scl_decode (min-sum f) or polar_scl_decode_boxplus (exact boxplus f, my_sn SCL_Dec)
  -> dict(u_info, u_packed, pm [B,L] fp64, list [B,L,words] int32)."""
  dev = tables.dev
  x = _prep_logits(logits, tables.n, dev)
  B, n, L = x.shape[0], tables.n, int(list_size)
  out = {"u_info": _out(dev, (B, tables.k), tc.float32, want_info),
         "u_packed": _out(dev, (B, words(n)), tc.int32, want_packed, out_packed),
         "pm": _out(dev, (B, L), tc.float64, want_pm),
         "list": _out(dev, (B, L, words(n)), tc.int32, want_list)}
  name = "polar_scl_decode" if not boxplus else (
    "polar_scl_decode_boxplus_pruned" if pruned else "polar_scl_decode_boxplus")   # pruned: use_fast_scl node shortcuts
  ws = "polar_scl_boxplus_workspace_bytes" if boxplus else "polar_scl_workspace_bytes"
  _call(dev, name, ptr(x), ptr(tables.frozen_mask), n, L, B, ptr(out["u_packed"]), ptr(out["u_info"]), ptr(tables.info_pos),
        tables.k, ptr(out["pm"]), ptr(out["list"]), ptr(crc_rows), int(crc_len), workspace=(ws, (n, L, B)))
  return out


HYBRID_MINSUM, HYBRID_BOXPLUS, HYBRID_BOXPLUS_PRUNED = 0, 1, 2


def scl_decode_hybrid(logits, tables, list_size, crc_rows, crc_len, cn_mode, want_info=True, want_packed=False,
                      out_packed=None, n_list_out=None):
  """polar_scl_decode_hybrid: SC on every row, CRC-aided list decoding (L paths) only of the rows whose SC decision fails
  the CRC.  cn_mode: HYBRID_MINSUM, HYBRID_BOXPLUS or HYBRID_BOXPLUS_PRUNED (both stages in that arithmetic).
  n_list_out: optional device int32 [1] tensor that receives the number of list-decoded rows (stream ordered).
  -> dict(u_info fp32 [B,k] | None, u_packed int32 [B,words] | None)."""
  dev = tables.dev
  x = _prep_logits(logits, tables.n, dev)
  B, n, L = x.shape[0], tables.n, int(list_size)
  out = {"u_info": _out(dev, (B, tables.k), tc.float32, want_info),
         "u_packed": _out(dev, (B, words(n)), tc.int32, want_packed, out_packed)}
  _call(dev, "polar_scl_decode_hybrid", ptr(x), ptr(tables.frozen_mask), n, L, B, ptr(out["u_packed"]), ptr(out["u_info"]),
        ptr(tables.info_pos), tables.k, ptr(crc_rows), int(crc_len), int(cn_mode), ptr(n_list_out),
        workspace=("polar_scl_hybrid_workspace_bytes", (n, L, B, int(cn_mode))))
  return out


def belief_decode(logits, tables, num_iter, boxplus, want_info=True, want_soft=False, want_packed=False, out_packed=None):
  """polar_belief_decode_f32: `num_iter` iterations of belief propagation with the min-sum or the exact boxplus f.
  -> dict(u_info fp32 [B,k] 0./1. | None, soft fp32 [B,k] logits at info_pos | None, u_packed int32 [B,words] | None).
  out_packed: caller-owned int32 [B, words(n)] buffer for the packed decisions (Monte-Carlo loop: no allocation per call)."""
  dev = tables.dev
  x = _prep_logits(logits, tables.n, dev)
  B = x.shape[0]
  out = {"u_info": _out(dev, (B, tables.k), tc.float32, want_info),
         "soft": _out(dev, (B, tables.k), tc.float32, want_soft),
         "u_packed": _out(dev, (B, words(tables.n)), tc.int32, want_packed, out_packed)}
  _call(dev, "polar_belief_decode_f32", ptr(x), ptr(tables.frozen_mask), tables.n, B, int(num_iter), 1 if boxplus else 0,
        ptr(out["u_packed"]), ptr(out["u_info"]), ptr(out["soft"]), ptr(tables.info_pos), tables.k)
  return out


def _host_logits(x, n):
  """CPU tensor -> contiguous fp32 [B, n] host tensor (no copy when it already is one)."""
  x = x.detach().reshape(-1, n)
  if x.dtype != tc.float32:
    x = x.to(tc.float32)
  return x.contiguous()


def sc_decode_host(logits_cpu, tables):
  """SC_Dec.forward on a CPU tensor: polar_sc_decode_host_f32 (chunked H2D -> decode -> D2H on two streams inside the call).
  Returns the [B, k] fp32 API tensor in page-locked host memory (torch's caching host allocator recycles it)."""
  x = _host_logits(logits_cpu, tables.n)
  B = x.shape[0]
  out = tc.empty((B, tables.k), dtype=tc.float32, pin_memory=B > 0)
  if B == 0:
    return out
  pos = tables.info_pos_np.astype(np.int32)
  check(lib().polar_sc_decode_host_f32(x.data_ptr(), tables.mask_np.ctypes.data, tables.n, B, None, out.data_ptr(),
                                       pos.ctypes.data, tables.k, init_device(tables.dev)))
  return out


def scl_decode_host(logits_cpu, tables, list_size, crc_rows_np=None, crc_len=0, want_pm=True):
  """SCL_Dec.forward on a CPU tensor: polar_scl_decode_host_f32.  -> (u_info [B,k] fp32 pinned, pm [B,L] fp64 | None)."""
  x = _host_logits(logits_cpu, tables.n)
  B, L = x.shape[0], int(list_size)
  out = tc.empty((B, tables.k), dtype=tc.float32, pin_memory=B > 0)
  pm = tc.empty((B, L), dtype=tc.float64, pin_memory=B > 0) if want_pm else None
  if B == 0:
    return out, pm
  pos = tables.info_pos_np.astype(np.int32)
  rows = None if crc_rows_np is None else np.ascontiguousarray(crc_rows_np, dtype=np.uint32)
  check(lib().polar_scl_decode_host_f32(x.data_ptr(), tables.mask_np.ctypes.data, tables.n, L, B, None, out.data_ptr(),
                                        pos.ctypes.data, tables.k, pm.data_ptr() if want_pm else None,
                                        rows.ctypes.data if rows is not None else None, int(crc_len), init_device(tables.dev)))
  return out, pm


def encode_f32(u, tables, want_packed=False):
  """polar_encode_f32: u [B,k] 0/1 -> c [B,n] fp32 (and optionally the packed codeword)."""
  dev = tables.dev
  u = u.to(device=dev, dtype=tc.float32).reshape(-1, tables.k).contiguous()
  B = u.shape[0]
  c = _out(dev, (B, tables.n), tc.float32)
  cp = _out(dev, (B, words(tables.n)), tc.int32, want_packed)
  _call(dev, "polar_encode_f32", ptr(u), ptr(tables.info_rank), tables.n, tables.k, B, ptr(c), ptr(cp))
  return (c, cp) if want_packed else c


def encode_packed(u_full_packed, n):
  x = u_full_packed.contiguous()
  out = tc.empty_like(x)
  _call(x.device, "polar_encode_packed", ptr(x), int(n), x.shape[0], ptr(out))
  return out


def _frontend_out(dev, B, n, e, want_codeword, out):
  """(u_packed int32 [B, words(n)], c_packed int32 [B, (e+31)//32] | None, logits fp32 [B, e]) of a front end;
  out = (u_packed, logits): caller-owned buffers (Monte-Carlo loop: no allocation per call)."""
  u, logit = out if out is not None else (None, None)
  return (_out(dev, (B, words(n)), tc.int32, given=u), _out(dev, (B, (e + 31) // 32), tc.int32, want_codeword),
          _out(dev, (B, e), tc.float32, given=logit))


def awgn_frontend(tables, batch_size, no, seed, offset=0, want_codeword=False, out=None):
  """polar_awgn_frontend -> (u_packed int32 [B,words], c_packed | None, logits fp32 [B,n]).
  out = (u_packed, logits): caller-owned buffers (Monte-Carlo loop: no allocation per call)."""
  dev, B, n = tables.dev, int(batch_size), tables.n
  u, c, logit = _frontend_out(dev, B, n, n, want_codeword, out)
  _call(dev, "polar_awgn_frontend", _philox_key(seed), int(offset), float(no), ptr(tables.frozen_mask), n, B, ptr(u), ptr(c),
        ptr(logit))
  return u, c, logit


def nr5g_awgn_frontend(plan, batch_size, no, seed, offset=0, want_codeword=False, out=None):
  """polar_nr5g_awgn_frontend for a device plan (NR5GPlan.on(dev)) -> (u_packed int32 [B, words(n)], c_packed int32
  [B, (e+31)//32] | None, logits fp32 [B, e]).  u_packed holds payload + CRC at their polar positions.
  out = (u_packed, logits): caller-owned buffers (Monte-Carlo loop: no allocation per call)."""
  dev, B, n, e = plan.dev, int(batch_size), plan.n, plan.e
  u, c, logit = _frontend_out(dev, B, n, e, want_codeword, out)
  _call(dev, "polar_nr5g_awgn_frontend", _philox_key(seed), int(offset), float(no), ptr(plan.payload_mask_d), ptr(plan.crc_rows_d),
        ptr(plan.crc_pos_d), plan.crc_len, ptr(plan.rm_idx_d), n, e, B, ptr(u), ptr(c), ptr(logit))
  return u, c, logit


def bec_frontend(tables, batch_size, pe, seed, offset=0, llr_max=100.0, want_codeword=False, out=None):
  """polar_bec_frontend -> (u_packed int32 [B,words], c_packed | None, logits fp32 [B,n] in {0, +-llr_max})."""
  dev, B, n = tables.dev, int(batch_size), tables.n
  u, c, logit = _frontend_out(dev, B, n, n, want_codeword, out)
  _call(dev, "polar_bec_frontend", _philox_key(seed), int(offset), float(pe), float(llr_max), ptr(tables.frozen_mask), n, B,
        ptr(u), ptr(c), ptr(logit))
  return u, c, logit


def bec_llr(c, pe, seed, offset=0, llr_max=100.0):
  c2 = _rows(c)
  out = tc.empty_like(c2)
  _call(c.device, "polar_bec_llr", _philox_key(seed), int(offset), float(pe), float(llr_max), ptr(c2), c2.shape[1], c2.shape[0],
        ptr(out))
  return out.reshape(c.shape)


def qpsk_awgn_llr(c, no, seed, offset=0):
  c2 = _rows(c)
  out = tc.empty_like(c2)
  _call(c.device, "polar_qpsk_awgn_llr", _philox_key(seed), int(offset), float(no), ptr(c2), c2.shape[1], c2.shape[0], ptr(out))
  return out.reshape(c.shape)


def unpack_info(packed, pos, n):
  dev = packed.device
  B, k = packed.shape[0], pos.shape[0]
  out = _out(dev, (B, k), tc.float32)
  _call(dev, "polar_unpack_info_f32", ptr(packed.contiguous()), ptr(pos), int(n), k, B, ptr(out))
  return out


def pack_bits(x):
  x2 = _rows(x)
  out = _out(x.device, (x2.shape[0], words(x2.shape[1])), tc.int32)
  _call(x.device, "polar_pack_bits_f32", ptr(x2), x2.shape[1], x2.shape[0], ptr(out))
  return out


def count_errors_f32(b, b_hat, counters):
  """counters: int64[2] device tensor, += (bit errors, block errors)."""
  dev = counters.device
  k = b.shape[-1]
  b2 = b.to(device=dev, dtype=tc.float32).reshape(-1, k).contiguous()
  h2 = b_hat.to(device=dev, dtype=tc.float32).reshape(-1, k).contiguous()
  _call(dev, "polar_count_errors_f32", ptr(b2), ptr(h2), k, b2.shape[0], ptr(counters))


def count_errors_packed(a, b, mask, n, counters):
  _call(counters.device, "polar_count_errors_packed", ptr(a.contiguous()), ptr(b.contiguous()), ptr(mask), int(n), a.shape[0],
        ptr(counters))


def gather_cols(x, idx):
  """polar_gather_cols_f32: out[b, e] = x[b, idx[e]] (idx int32 device tensor)."""
  x2 = _rows(x)
  out = _out(x.device, (x2.shape[0], idx.shape[0]), tc.float32)
  _call(x.device, "polar_gather_cols_f32", ptr(x2), ptr(idx), x2.shape[1], idx.shape[0], x2.shape[0], ptr(out))
  return out


def rate_recover(x, src0, src1, fill, out=None):
  """polar_rate_recover_f32: out[b, j] = (src0[j] >= 0 ? x[b, src0[j]] : fill[j]) + (src1[j] >= 0 ? x[b, src1[j]] : 0).
  out: optional caller-owned fp32 [B, len(src0)] buffer."""
  x2 = _rows(x)
  out = _out(x.device, (x2.shape[0], src0.shape[0]), tc.float32, given=out)
  _call(x.device, "polar_rate_recover_f32", ptr(x2), ptr(src0), ptr(src1), ptr(fill), x2.shape[1], src0.shape[0],
        x2.shape[0], ptr(out))
  return out


MC_GROUP_MAX = 32


def mc_control_group(delta, item_points, state, sweep, expect_q, target_bit_errs, target_block_errs, max_mc_iter, early_stop):
  """polar_mc_control_group: fold the counters delta [G,4] of a group of queued iterations (SNR point of iteration j =
  item_points[j]) into the per-point states [P,8] and the sweep cursor [8], with sim_ber's stop rules, on the device."""
  pts = (ctypes.c_int32 * len(item_points))(*[int(p) for p in item_points])
  _call(state.device, "polar_mc_control_group", ptr(delta), ctypes.cast(pts, ctypes.c_void_p), len(item_points), ptr(state),
        state.shape[0], ptr(sweep), int(expect_q), _stop_target(target_bit_errs), _stop_target(target_block_errs), int(max_mc_iter),
        1 if early_stop else 0)


def osd_decode(logits, gm_rows, n, k, t, want_f32=True, want_packed=False, want_dist=False):
  """polar_osd_decode: logits [B,n] + bit-packed generator rows (device int32 [k, words]) -> dict(c fp32 [B,n], c_packed, dist)."""
  dev = gm_rows.device
  x = _prep_logits(logits, n, dev)
  B = x.shape[0]
  out = {"c": _out(dev, (B, n), tc.float32, want_f32),
         "c_packed": _out(dev, (B, (n + 31) // 32), tc.int32, want_packed),
         "dist": _out(dev, (B,), tc.float32, want_dist)}
  _call(dev, "polar_osd_decode", ptr(x), ptr(gm_rows), n, k, int(t), B, ptr(out["c_packed"]), ptr(out["c"]), ptr(out["dist"]))
  return out


def launch_count():
  return int(lib().polar_launch_count())
