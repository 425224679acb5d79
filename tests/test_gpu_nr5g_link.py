"""5G NR polar codes in the fused AWGN link model: the front end `polar_nr5g_awgn_frontend` (payload -> CRC -> channel
allocation -> polar transform -> rate matching -> QPSK/AWGN -> demapper in one launch), the plan it runs from
(`Polar5GEncoder.frontend_plan`), `Polar5GDecoder.decode_packed` and the on-device Monte-Carlo loop counting payload
bits of a rate-matched code.  The CPU tests restate the kernel's bit path in numpy against the golden codewords of the
reference; the GPU tests check the kernel bit for bit against the layer composition and the device loop counter for
counter against the host loop."""
import ctypes

import numpy as np
import pytest

from util import golden, unpack_words

# (k, E): none / puncturing / shortening / repetition, CRC6 and CRC11, E % 4 in {0, 1, 2, 3}
CODES = [(64, 128), (100, 300), (200, 400), (300, 1088), (16, 61), (40, 70), (30, 101), (30, 103)]


def _plan_bit_path(plan, payload):
    """numpy restatement of the kernel's bit path: payload [B, k] -> (u [B, n] with payload + CRC, rate-matched c [B, e])."""
    from oracle import polar_oracle as po
    B = payload.shape[0]
    u = np.zeros((B, plan.n), dtype=np.uint8)
    u[:, plan.payload_pos] = payload
    rows = plan.crc_rows[plan.payload_pos]                              # generator word of payload bit t
    bits = (rows[:, None] >> np.arange(plan.crc_len - 1, -1, -1, dtype=np.uint32)[None, :]) & 1   # [k, crc_len], MSB = bit 0
    u[:, plan.crc_pos] = (payload.astype(np.int64) @ bits.astype(np.int64)) % 2
    return u, po.polar_transform(u)[:, plan.rm_idx]


def test_frontend_plan_reproduces_golden_codewords():
    from my_sn.fec.polar.enc import Polar5GEncoder
    g = golden("nr5g")
    for k, e in g["cfgs"]:
        key = "%d_%d" % (k, e)
        enc = Polar5GEncoder(int(k), int(e))
        plan = enc.frontend_plan()
        assert (plan.n, plan.e, plan.k, plan.crc_len) == (int(g["npolar_" + key]), e, k, int(g["crclen_" + key]))
        assert np.array_equal(plan.rm_idx, g["idx_" + key])
        _, c = _plan_bit_path(plan, g["u_" + key])
        assert np.array_equal(c, g["c_" + key]), key
        assert enc.frontend_plan() is plan                              # built once


@pytest.mark.parametrize("k,e", CODES)
def test_frontend_plan_consistency(k, e):
    from my_sn.fec.polar.enc import Polar5GEncoder
    enc = Polar5GEncoder(k, e)
    plan = enc.frontend_plan()
    n = plan.n
    assert n == enc.n_polar and plan.e == e and plan.k == k and plan.crc_len == enc.enc_crc.crc_length
    mask = unpack_words(plan.payload_mask[None, :], n)[0]
    assert mask.sum() == k and np.array_equal(np.nonzero(mask)[0], plan.payload_pos)
    sets = [set(plan.payload_pos.tolist()), set(plan.crc_pos.tolist()), set(np.asarray(enc.frozen_pos).tolist())]
    assert sum(len(s) for s in sets) == n and set().union(*sets) == set(range(n))
    assert not (plan.crc_rows[np.setdiff1d(np.arange(n), plan.payload_pos)]).any()
    assert plan.rm_idx.min() >= 0 and plan.rm_idx.max() < n and plan.rm_idx.shape == (e,)


def test_downlink_plan_raises_and_link_model_checks():
    import torch
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    from z_sys_model.awgn_model import System_AWGN_model
    with pytest.raises(Exception):
        Polar5GEncoder(30, 108, channel_type="downlink").frontend_plan()
    enc = Polar5GEncoder(100, 300)
    dec = Polar5GDecoder(enc, "SCL")
    with pytest.raises(AssertionError):
        System_AWGN_model(512, 100, enc, dec)
    with pytest.raises(AssertionError):
        System_AWGN_model(300, 111, enc, dec)
    with pytest.raises(ValueError):
        System_AWGN_model(300, 100, enc, dec, cw_estimates=True)
    m = System_AWGN_model(300, 100, enc, dec)
    assert m.coderate == 100 / 300
    System_AWGN_model(300, 100, enc, dec, cw_estimates=True, fused=False)


def test_argument_checks_without_gpu():
    import d_kernels as dk
    lib = dk.lib()
    d = 256                                                             # never dereferenced: every call below fails early

    def call(n=128, e=128, crc_len=11, B=5, no=0.5, pm=d, rows=d, pos=d, idx=d, u=d, lg=d):
        return lib.polar_nr5g_awgn_frontend(1, 0, no, pm, rows, pos, crc_len, idx, n, e, B, u, None, lg, None)
    before = lib.polar_launch_count()
    for kw in (dict(n=16), dict(n=48), dict(n=2048), dict(e=0), dict(e=8193), dict(crc_len=0), dict(crc_len=33),
               dict(B=-1), dict(no=0.0), dict(no=-1.0), dict(no=float("nan")), dict(pm=None), dict(rows=None),
               dict(pos=None), dict(idx=None), dict(u=None), dict(lg=None)):
        assert call(**kw) == dk.POLAR_EINVAL, kw
    assert call(B=0, u=None, lg=None) == dk.POLAR_OK
    assert lib.polar_launch_count() == before


# ---------------------------------------------------------------------------------------------------------------------
def _env():
    import torch
    import d_kernels as dk
    from oracle import polar_oracle as po
    return torch, dk, po, torch.device("cuda", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("k,e", CODES)
def test_kernel_equals_composition(k, e):
    torch, dk, po, dev = _env()
    from my_sn.fec.crc import CRCEncoder
    from my_sn.fec.polar.enc import Polar5GEncoder
    enc = Polar5GEncoder(k, e)
    plan = enc.frontend_plan(dev)
    n = plan.n
    B, seed, off = 20000, 1234, 77                                      # > one codeword per warp of the persistent grid
    no = po.ebnodb2no(2.0, 2, k / e)
    u, c, lg = dk.nr5g_awgn_frontend(plan, B, no, seed, off, want_codeword=True)
    assert u.shape == (B, dk.words(n)) and c.shape == (B, (e + 31) // 32) and lg.shape == (B, e)
    ub = unpack_words(u.cpu().numpy(), n)
    payload = ub[:, plan.payload_pos]
    assert abs(payload.mean() - 0.5) < 5 * 0.5 / np.sqrt(B * k)
    assert not ub[:, np.asarray(enc.frozen_pos)].any()
    crc = CRCEncoder(enc.enc_crc.crc_degree, k)(torch.from_numpy(payload.astype(np.float32)))[:, k:]
    assert np.array_equal(ub[:, plan.crc_pos], crc.numpy().astype(np.uint8))
    c_ref = enc(torch.from_numpy(payload.astype(np.float32)).to(dev))   # CRC + polar transform + rate-matching gather
    words = unpack_words(c.cpu().numpy(), 32 * c.shape[1])
    assert np.array_equal(words[:, :e], c_ref.cpu().numpy().astype(np.uint8)) and not words[:, e:].any()
    e4 = (e + 3) // 4 * 4
    cpad = torch.zeros((B, e4), dtype=torch.float32, device=dev)
    cpad[:, :e] = c_ref
    assert torch.equal(lg, dk.qpsk_awgn_llr(cpad, no, seed, off)[:, :e])
    # counter-based stream: codeword b at offset o is codeword b-1 at offset o+1
    u2, _, lg2 = dk.nr5g_awgn_frontend(plan, B - 1, no, seed, off + 1)
    assert torch.equal(u2, u[1:]) and torch.equal(lg2, lg[1:])
    # caller-owned buffers, 16-byte aligned rows and rows shifted by one float
    for shift in (0, 1):
        flat = torch.full((B * e + 4,), float("nan"), dtype=torch.float32, device=dev)
        lo = flat[shift:shift + B * e].view(B, e)
        uo = torch.full_like(u, -1)
        dk.nr5g_awgn_frontend(plan, B, no, seed, off, out=(uo, lo))
        assert torch.equal(uo, u) and torch.equal(lo, lg), shift
        assert torch.isnan(flat[:shift]).all() and torch.isnan(flat[shift + B * e:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("k,e", [(64, 128), (100, 300), (200, 400), (300, 1088), (16, 61), (30, 103)])
def test_noiseless_link_decodes_every_payload(k, e):
    torch, dk, po, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    from z_sys_model.awgn_model import System_AWGN_model
    enc = Polar5GEncoder(k, e)
    for kind in ("SC", "SCL", "hybSCL"):
        model = System_AWGN_model(e, k, enc, Polar5GDecoder(enc, kind, list_size=8), seed=5)
        bits, bits_hat = model(batch_size=2000, ebno_db=40.0)
        assert bits.shape == (2000, k) and bits_hat.shape == (2000, k) and bits.is_cuda
        assert torch.equal(bits, bits_hat), kind
        assert model._offset == 2000


@pytest.mark.gpu
def test_fused_bler_inside_confidence_band_of_layer_path():
    torch, dk, po, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    from z_sys_model.awgn_model import System_AWGN_model
    k, e, bs, iters = 100, 300, 10000, 3
    enc = Polar5GEncoder(k, e)
    torch.manual_seed(11)
    for ebno in (1.0, 2.0):
        bler = {}
        for fused in (True, False):
            model = System_AWGN_model(e, k, enc, Polar5GDecoder(enc, "SCL", list_size=8), fused=fused, seed=21)
            errs = 0
            for _ in range(iters):
                b, bh = model(batch_size=bs, ebno_db=ebno)
                assert b.shape == (bs, k) and bh.shape == (bs, k)
                errs += int((b.to(dev) != bh.to(dev)).any(-1).sum())
            bler[fused] = errs / (bs * iters)
        p = 0.5 * (bler[True] + bler[False])
        band = 5 * np.sqrt(max(p * (1 - p), 1e-4) * 2 / (bs * iters))
        assert abs(bler[True] - bler[False]) < band, (ebno, bler)


_STOP_CASES = (dict(max_mc_iter=7, target_block_errs=500), dict(max_mc_iter=5, target_bit_errs=2000),
               dict(max_mc_iter=3), dict(max_mc_iter=1, target_block_errs=1))


@pytest.mark.gpu
@pytest.mark.parametrize("k,e", [(100, 300), (40, 70)])
@pytest.mark.parametrize("kind", ["SC", "SCL", "hybSCL"])
def test_device_loop_equals_host_loop(kind, k, e, monkeypatch):
    torch, dk, po, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    from z_sys_model.awgn_model import System_AWGN_model
    import my_sn.sim as sim
    enc = Polar5GEncoder(k, e)
    mk = lambda seed: System_AWGN_model(e, k, enc, Polar5GDecoder(enc, kind, list_size=8), seed=seed)
    ebnos = np.array([-1.0, 1.0, 2.5, 4.0, 9.0, 10.0], dtype=np.float32)
    bs = 3000
    for kw in _STOP_CASES:
        host, devm = mk(99), mk(99)
        ber_h, bler_h = sim.sim_ber(host, ebnos, bs, verbose=False, on_device=False, **kw)
        ber_d, bler_d, cnt, status, iters = sim.sim_ber_device(devm, ebnos, bs, verbose=False, return_counters=True, **kw)
        assert torch.equal(ber_h, ber_d) and torch.equal(bler_h, bler_d), (kind, kw)
        assert host._offset == devm._offset
        assert (iters <= kw["max_mc_iter"]).all() and int(status[0]) in (1, 3, 4)
        assert (cnt[:, 2] == cnt[:, 3] * k).all()                       # counted bits are payload bits
        if "target_block_errs" in kw and cnt[0, 1] >= kw["target_block_errs"]:
            assert status[0] == 4
        if "target_bit_errs" in kw and cnt[0, 0] >= kw["target_bit_errs"]:
            assert status[0] == 3
        zero = np.nonzero((cnt[:, 1] == 0) & (cnt[:, 3] > 0))[0]
        if len(zero):
            assert status[zero[0]] == 2 and (cnt[zero[0] + 1:] == 0).all()
    # a model built as in the reference goes to the device loop by default
    calls = []
    real = sim.sim_ber_device
    monkeypatch.setattr(sim, "sim_ber_device", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    a, b = mk(5), mk(5)
    r1 = sim.sim_ber(a, ebnos[:3], bs, 2, verbose=False)
    assert calls == [1]
    r2 = sim.sim_ber(b, ebnos[:3], bs, 2, verbose=False, on_device=False)
    assert calls == [1] and torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1]) and a._offset == b._offset


@pytest.mark.gpu
def test_device_loop_with_process_group_of_one():
    torch, dk, po, dev = _env()
    import torch.distributed as dist
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    from z_sys_model.awgn_model import System_AWGN_model
    from my_sn.sim import sim_ber_device
    k, e, bs = 200, 400, 2000
    enc = Polar5GEncoder(k, e)
    ebnos = np.array([1.0, 2.0, 3.0], dtype=np.float32)
    mk = lambda: System_AWGN_model(e, k, enc, Polar5GDecoder(enc, "SCL", list_size=8), seed=3)
    ref = sim_ber_device(mk(), ebnos, bs, 3, target_block_errs=100, verbose=False, return_counters=True)
    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1)
    try:
        got = sim_ber_device(mk(), ebnos, bs, 3, target_block_errs=100, verbose=False, return_counters=True)
    finally:
        dist.destroy_process_group()
    assert np.array_equal(ref[2], got[2]) and np.array_equal(ref[3], got[3]) and np.array_equal(ref[4], got[4])
    assert ref[2][:, 3].sum() > 0
