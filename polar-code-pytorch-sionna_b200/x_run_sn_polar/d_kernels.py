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
SC_MAX_N, SCL_MAX_N, SCL_MAX_L = 8192, 4096, 32

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
  "polar_mc_control": (_i32, [_vp, _vp, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong, _vp]),
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


def frozen_mask_words(frozen_pos, n):
  """uint32[words(n)]: bit (i % 32) of word (i // 32) set <=> position i frozen (as int32 bit pattern)."""
  f = np.zeros(max(n, 32), dtype=np.uint8)
  f[to_numpy_pos(frozen_pos)] = 1
  w = np.packbits(f.reshape(-1, 32), axis=1, bitorder="little").view(np.uint32).reshape(-1)
  return w[:words(n)].copy()


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
    self.frozen_mask = tc.from_numpy(self.mask_np.view(np.int32).copy()).to(dev)
    self.info_pos = tc.from_numpy(self.info_pos_np.astype(np.int32)).to(dev)
    self.info_rank = tc.from_numpy(rank).to(dev)
    info_mask = (~self.mask_np) & (np.uint32(0xFFFFFFFF) if self.n >= 32 else np.uint32((1 << self.n) - 1))
    self.info_mask = tc.from_numpy(np.asarray(info_mask, dtype=np.uint32).view(np.int32).copy()).to(dev)


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
    f = np.zeros(max(self.n, 32), dtype=np.uint8)
    f[self.payload_pos] = 1
    self.payload_mask = np.packbits(f.reshape(-1, 32), axis=1, bitorder="little").view(np.uint32).reshape(-1)[:words(self.n)].copy()
    self.dev = None
    self._on = {}

  def on(self, dev):
    p = self._on.get(str(dev))
    if p is None:
      init_device(dev)
      p = self._on[str(dev)] = copy.copy(self)
      p.dev, p._on = dev, None
      i32 = lambda a: tc.from_numpy(np.ascontiguousarray(a).astype(np.int64).astype(np.int32)).to(dev)
      p.payload_mask_d = tc.from_numpy(self.payload_mask.view(np.int32).copy()).to(dev)
      p.crc_rows_d = tc.from_numpy(self.crc_rows.view(np.int32).copy()).to(dev)
      p.crc_pos_d, p.rm_idx_d, p.payload_pos_d = i32(self.crc_pos), i32(self.rm_idx), i32(self.payload_pos)
    return p


_TABLE_CACHE = {}


def code_tables(frozen_pos, n, dev):
  key = (to_numpy_pos(frozen_pos).tobytes(), int(n), str(dev))
  tb = _TABLE_CACHE.get(key)
  if tb is None:
    tb = _TABLE_CACHE[key] = CodeTables(frozen_pos, n, dev)
  return tb


# ---- kernel wrappers (device tensors in, device tensors out) -------------------------------------------
def _prep_logits(x, n, dev):
  x = x.to(device=dev, dtype=tc.float32).reshape(-1, n)
  if not x.is_contiguous() or x.data_ptr() % 16:
    x = x.contiguous().clone() if x.data_ptr() % 16 else x.contiguous()
  return x


def sc_decode(logits, tables, want_info=True, want_packed=False, boxplus=False, out_packed=None):
  """polar_sc_decode_f32 (min-sum f) or polar_sc_decode_boxplus_f32 (exact boxplus f, my_sn SC_Dec).
  logits [B,n] (any float dtype/device) -> (u_info fp32 [B,k] | None, u_packed int32 | None).
  out_packed: caller-owned int32 [B, words(n)] buffer for the packed decisions (Monte-Carlo loop: no allocation per call)."""
  dev = tables.dev
  x = _prep_logits(logits, tables.n, dev)
  B = x.shape[0]
  u_info = tc.empty((B, tables.k), dtype=tc.float32, device=dev) if want_info else None
  u_packed = out_packed if out_packed is not None else (
    tc.empty((B, words(tables.n)), dtype=tc.int32, device=dev) if want_packed else None)
  with tc.cuda.device(dev):
    fn = lib().polar_sc_decode_boxplus_f32 if boxplus else lib().polar_sc_decode_f32
    check(fn(ptr(x), ptr(tables.frozen_mask), tables.n, B, ptr(u_packed), ptr(u_info), ptr(tables.info_pos), tables.k,
             stream_ptr(dev)))
  return u_info, u_packed


_WS_CACHE = {}


def scl_decode(logits, tables, list_size, crc_rows=None, crc_len=0, want_info=True, want_packed=False,
               want_pm=False, want_list=False, boxplus=False, out_packed=None, pruned=False):
  """polar_scl_decode (min-sum f) or polar_scl_decode_boxplus (exact boxplus f, my_sn SCL_Dec)
  -> dict(u_info, u_packed, pm [B,L] fp64, list [B,L,words] int32)."""
  dev = tables.dev
  x = _prep_logits(logits, tables.n, dev)
  B, n, L = x.shape[0], tables.n, int(list_size)
  out = {"u_info": None, "u_packed": None, "pm": None, "list": None}
  if want_info:
    out["u_info"] = tc.empty((B, tables.k), dtype=tc.float32, device=dev)
  if out_packed is not None:
    out["u_packed"] = out_packed
  elif want_packed:
    out["u_packed"] = tc.empty((B, words(n)), dtype=tc.int32, device=dev)
  if want_pm:
    out["pm"] = tc.empty((B, L), dtype=tc.float64, device=dev)
  if want_list:
    out["list"] = tc.empty((B, L, words(n)), dtype=tc.int32, device=dev)
  with tc.cuda.device(dev):
    fn_ws = lib().polar_scl_boxplus_workspace_bytes if boxplus else lib().polar_scl_workspace_bytes
    fn_dec = lib().polar_scl_decode if not boxplus else (
      lib().polar_scl_decode_boxplus_pruned if pruned else lib().polar_scl_decode_boxplus)   # pruned: use_fast_scl node shortcuts
    need = int(fn_ws(n, L, B)) if B > 0 else 0
    ws = _workspace(dev, need)
    check(fn_dec(ptr(x), ptr(tables.frozen_mask), n, L, B, ptr(out["u_packed"]), ptr(out["u_info"]),
                                 ptr(tables.info_pos), tables.k, ptr(out["pm"]), ptr(out["list"]),
                                 ptr(crc_rows), int(crc_len), ptr(ws), need, stream_ptr(dev)))
  return out


def _workspace(dev, need):
  """The per-device list-decoder workspace (grown, never shrunk), or None when `need` is 0."""
  if not need:
    return None
  ws = _WS_CACHE.get(str(dev))
  if ws is None or ws.numel() < need:
    ws = _WS_CACHE[str(dev)] = tc.empty(need + 256, dtype=tc.uint8, device=dev)
  return ws


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
  out = {"u_info": tc.empty((B, tables.k), dtype=tc.float32, device=dev) if want_info else None,
         "u_packed": out_packed if out_packed is not None else (
           tc.empty((B, words(n)), dtype=tc.int32, device=dev) if want_packed else None)}
  with tc.cuda.device(dev):
    need = int(lib().polar_scl_hybrid_workspace_bytes(n, L, B, int(cn_mode))) if B > 0 else 0
    ws = _workspace(dev, need)
    check(lib().polar_scl_decode_hybrid(ptr(x), ptr(tables.frozen_mask), n, L, B, ptr(out["u_packed"]), ptr(out["u_info"]),
                                        ptr(tables.info_pos), tables.k, ptr(crc_rows), int(crc_len), int(cn_mode),
                                        ptr(n_list_out), ptr(ws), need, stream_ptr(dev)))
  return out


def _host_logits(x, n):
  """CPU tensor -> contiguous fp32 [B, n] host tensor (no copy when it already is one)."""
  x = x.detach().reshape(-1, n)
  if x.dtype != tc.float32:
    x = x.to(tc.float32)
  return x.contiguous()


def sc_decode_host(logits_cpu, tables, boxplus=False):
  """SC_Dec.forward on a CPU tensor: polar_sc_decode_host_f32 (chunked H2D -> decode -> D2H on two streams inside the call).
  Returns the [B, k] fp32 API tensor in page-locked host memory (torch's caching host allocator recycles it)."""
  if boxplus:      # the boxplus decoders have no host-buffer entry point: plain copy, decode, copy back
    u, _ = sc_decode(logits_cpu, tables, want_info=True, boxplus=True)
    return u.cpu()
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
  c = tc.empty((B, tables.n), dtype=tc.float32, device=dev)
  cp = tc.empty((B, words(tables.n)), dtype=tc.int32, device=dev) if want_packed else None
  with tc.cuda.device(dev):
    check(lib().polar_encode_f32(ptr(u), ptr(tables.info_rank), tables.n, tables.k, B, ptr(c), ptr(cp), stream_ptr(dev)))
  return (c, cp) if want_packed else c


def encode_packed(u_full_packed, n):
  dev = u_full_packed.device
  x = u_full_packed.contiguous()
  out = tc.empty_like(x)
  with tc.cuda.device(dev):
    check(lib().polar_encode_packed(ptr(x), int(n), x.shape[0], ptr(out), stream_ptr(dev)))
  return out


def awgn_frontend(tables, batch_size, no, seed, offset=0, want_codeword=False, out=None):
  """polar_awgn_frontend -> (u_packed int32 [B,words], c_packed | None, logits fp32 [B,n]).
  out = (u_packed, logits): caller-owned buffers (Monte-Carlo loop: no allocation per call)."""
  dev = tables.dev
  B, n = int(batch_size), tables.n
  u = out[0] if out is not None else tc.empty((B, words(n)), dtype=tc.int32, device=dev)
  c = tc.empty((B, words(n)), dtype=tc.int32, device=dev) if want_codeword else None
  logit = out[1] if out is not None else tc.empty((B, n), dtype=tc.float32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_awgn_frontend(int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset), float(no), ptr(tables.frozen_mask), n, B,
                                    ptr(u), ptr(c), ptr(logit), stream_ptr(dev)))
  return u, c, logit


def nr5g_awgn_frontend(plan, batch_size, no, seed, offset=0, want_codeword=False, out=None):
  """polar_nr5g_awgn_frontend for a device plan (NR5GPlan.on(dev)) -> (u_packed int32 [B, words(n)], c_packed int32
  [B, (e+31)//32] | None, logits fp32 [B, e]).  u_packed holds payload + CRC at their polar positions.
  out = (u_packed, logits): caller-owned buffers (Monte-Carlo loop: no allocation per call)."""
  dev = plan.dev
  B, n, e = int(batch_size), plan.n, plan.e
  u = out[0] if out is not None else tc.empty((B, words(n)), dtype=tc.int32, device=dev)
  c = tc.empty((B, (e + 31) // 32), dtype=tc.int32, device=dev) if want_codeword else None
  logit = out[1] if out is not None else tc.empty((B, e), dtype=tc.float32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_nr5g_awgn_frontend(int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset), float(no), ptr(plan.payload_mask_d),
                                         ptr(plan.crc_rows_d), ptr(plan.crc_pos_d), plan.crc_len, ptr(plan.rm_idx_d), n, e, B,
                                         ptr(u), ptr(c), ptr(logit), stream_ptr(dev)))
  return u, c, logit


def bec_frontend(tables, batch_size, pe, seed, offset=0, llr_max=100.0, want_codeword=False, out=None):
  """polar_bec_frontend -> (u_packed int32 [B,words], c_packed | None, logits fp32 [B,n] in {0, +-llr_max})."""
  dev = tables.dev
  B, n = int(batch_size), tables.n
  u = out[0] if out is not None else tc.empty((B, words(n)), dtype=tc.int32, device=dev)
  c = tc.empty((B, words(n)), dtype=tc.int32, device=dev) if want_codeword else None
  logit = out[1] if out is not None else tc.empty((B, n), dtype=tc.float32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_bec_frontend(int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset), float(pe), float(llr_max),
                                   ptr(tables.frozen_mask), n, B, ptr(u), ptr(c), ptr(logit), stream_ptr(dev)))
  return u, c, logit


def bec_llr(c, pe, seed, offset=0, llr_max=100.0):
  dev = c.device
  c2 = c.to(tc.float32).reshape(-1, c.shape[-1]).contiguous()
  out = tc.empty_like(c2)
  with tc.cuda.device(dev):
    check(lib().polar_bec_llr(int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset), float(pe), float(llr_max), ptr(c2), c2.shape[1],
                              c2.shape[0], ptr(out), stream_ptr(dev)))
  return out.reshape(c.shape)


def qpsk_awgn_llr(c, no, seed, offset=0):
  dev = c.device
  c2 = c.to(tc.float32).reshape(-1, c.shape[-1]).contiguous()
  out = tc.empty_like(c2)
  with tc.cuda.device(dev):
    check(lib().polar_qpsk_awgn_llr(int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset), float(no), ptr(c2), c2.shape[1], c2.shape[0],
                                    ptr(out), stream_ptr(dev)))
  return out.reshape(c.shape)


def unpack_info(packed, pos, n):
  dev = packed.device
  B, k = packed.shape[0], pos.shape[0]
  out = tc.empty((B, k), dtype=tc.float32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_unpack_info_f32(ptr(packed.contiguous()), ptr(pos), int(n), k, B, ptr(out), stream_ptr(dev)))
  return out


def pack_bits(x):
  dev = x.device
  x2 = x.to(tc.float32).reshape(-1, x.shape[-1]).contiguous()
  out = tc.empty((x2.shape[0], words(x2.shape[1])), dtype=tc.int32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_pack_bits_f32(ptr(x2), x2.shape[1], x2.shape[0], ptr(out), stream_ptr(dev)))
  return out


def count_errors_f32(b, b_hat, counters):
  """counters: int64[2] device tensor, += (bit errors, block errors)."""
  dev = counters.device
  k = b.shape[-1]
  b2 = b.to(device=dev, dtype=tc.float32).reshape(-1, k).contiguous()
  h2 = b_hat.to(device=dev, dtype=tc.float32).reshape(-1, k).contiguous()
  with tc.cuda.device(dev):
    check(lib().polar_count_errors_f32(ptr(b2), ptr(h2), k, b2.shape[0], ptr(counters), stream_ptr(dev)))


def count_errors_packed(a, b, mask, n, counters):
  dev = counters.device
  with tc.cuda.device(dev):
    check(lib().polar_count_errors_packed(ptr(a.contiguous()), ptr(b.contiguous()), ptr(mask), int(n), a.shape[0],
                                          ptr(counters), stream_ptr(dev)))


def gather_cols(x, idx):
  """polar_gather_cols_f32: out[b, e] = x[b, idx[e]] (idx int32 device tensor)."""
  dev = x.device
  x2 = x.to(tc.float32).reshape(-1, x.shape[-1]).contiguous()
  out = tc.empty((x2.shape[0], idx.shape[0]), dtype=tc.float32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_gather_cols_f32(ptr(x2), ptr(idx), x2.shape[1], idx.shape[0], x2.shape[0], ptr(out), stream_ptr(dev)))
  return out


def rate_recover(x, src0, src1, fill, out=None):
  """polar_rate_recover_f32: out[b, j] = (src0[j] >= 0 ? x[b, src0[j]] : fill[j]) + (src1[j] >= 0 ? x[b, src1[j]] : 0).
  out: optional caller-owned fp32 [B, len(src0)] buffer."""
  dev = x.device
  x2 = x.to(tc.float32).reshape(-1, x.shape[-1]).contiguous()
  if out is None:
    out = tc.empty((x2.shape[0], src0.shape[0]), dtype=tc.float32, device=dev)
  with tc.cuda.device(dev):
    check(lib().polar_rate_recover_f32(ptr(x2), ptr(src0), ptr(src1), ptr(fill), x2.shape[1], src0.shape[0], x2.shape[0],
                                       ptr(out), stream_ptr(dev)))
  return out


def mc_control(delta, state, target_bit_errs, target_block_errs, max_mc_iter):
  """polar_mc_control: fold `delta` (int64[4]) into `state` (int64[8]) and evaluate sim_ber's stop rules on the device."""
  dev = state.device
  tb = -1 if target_bit_errs is None else int(target_bit_errs)
  tk = -1 if target_block_errs is None else int(target_block_errs)
  with tc.cuda.device(dev):
    check(lib().polar_mc_control(ptr(delta), ptr(state), tb, tk, int(max_mc_iter), stream_ptr(dev)))


MC_GROUP_MAX = 32


def mc_control_group(delta, item_points, state, sweep, expect_q, target_bit_errs, target_block_errs, max_mc_iter, early_stop):
  """polar_mc_control_group: fold the counters delta [G,4] of a group of queued iterations (SNR point of iteration j =
  item_points[j]) into the per-point states [P,8] and the sweep cursor [8], with sim_ber's stop rules, on the device."""
  dev = state.device
  tb = -1 if target_bit_errs is None else int(target_bit_errs)
  tk = -1 if target_block_errs is None else int(target_block_errs)
  pts = (ctypes.c_int32 * len(item_points))(*[int(p) for p in item_points])
  with tc.cuda.device(dev):
    check(lib().polar_mc_control_group(ptr(delta), ctypes.cast(pts, ctypes.c_void_p), len(item_points), ptr(state), state.shape[0],
                                       ptr(sweep), int(expect_q), tb, tk, int(max_mc_iter), 1 if early_stop else 0, stream_ptr(dev)))


def pack_rows(m):
  """0/1 matrix [r, n] (numpy) -> uint32 bit-packed rows [r, (n+31)//32], position i = bit i%32 of word i//32 (as int32)."""
  m = (np.asarray(m) != 0).astype(np.uint8)
  r, n = m.shape
  nw = (n + 31) // 32
  pad = np.zeros((r, nw * 32), dtype=np.uint8)
  pad[:, :n] = m
  return np.packbits(pad.reshape(r, nw, 32), axis=2, bitorder="little").view(np.uint32).reshape(r, nw).view(np.int32).copy()


def osd_decode(logits, gm_rows, n, k, t, want_f32=True, want_packed=False, want_dist=False):
  """polar_osd_decode: logits [B,n] + bit-packed generator rows (device int32 [k, words]) -> dict(c fp32 [B,n], c_packed, dist)."""
  dev = gm_rows.device
  x = _prep_logits(logits, n, dev)
  B = x.shape[0]
  nw = (n + 31) // 32
  out = {"c": tc.empty((B, n), dtype=tc.float32, device=dev) if want_f32 else None,
         "c_packed": tc.empty((B, nw), dtype=tc.int32, device=dev) if want_packed else None,
         "dist": tc.empty((B,), dtype=tc.float32, device=dev) if want_dist else None}
  with tc.cuda.device(dev):
    check(lib().polar_osd_decode(ptr(x), ptr(gm_rows), n, k, int(t), B, ptr(out["c_packed"]), ptr(out["c"]), ptr(out["dist"]),
                                 stream_ptr(dev)))
  return out


def launch_count():
  return int(lib().polar_launch_count())
