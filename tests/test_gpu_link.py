"""GPU tests of the pieces either side of the decoders: AWGN front end (statistical parity: the
reference draws from torch's CPU mt19937, the kernel from Philox), error counters, CRC-aided list
decoding, the link model + Monte-Carlo loop (BER/BLER inside confidence intervals of the oracle),
and the host-buffer C-ABI entry points."""
import numpy as np
import pytest

from util import golden, golden_names, unpack_words, pack_words, awgn_logits, set_opt

pytestmark = pytest.mark.gpu


def _env():
    import torch
    import d_kernels as dk
    from oracle import polar_oracle as po, c_oracle as co
    return torch, dk, po, co, torch.device("cuda", 0)


@pytest.mark.parametrize("n,k", [(8, 4), (32, 16), (64, 32), (1024, 512), (4096, 2048)])
def test_frontend_structure_and_statistics(n, k):
    torch, dk, po, co, dev = _env()
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    B = max(4096, (1 << 21) // n)
    ebno = 2.0
    no = po.ebnodb2no(ebno, 2, k / n)
    u, c, lg = dk.awgn_frontend(tables, B, no, seed=99, offset=5, want_codeword=True)
    ub = unpack_words(u.cpu().numpy(), n)
    cb = unpack_words(c.cpu().numpy(), n)
    assert not ub[:, fp].any()                                         # frozen positions carry 0 (enc.py:33-35)
    assert abs(ub[:, po.info_positions(fp, n)].mean() - 0.5) < 5 * 0.5 / np.sqrt(B * k)   # Bernoulli(1/2) source
    assert np.array_equal(co.polar_transform(ub), cb)                  # codeword = u.G
    y = lg.cpu().numpy().astype(np.float64) * (-no / (2 * np.sqrt(2)))   # invert the closed-form demapper
    z = (y - (1 - 2.0 * cb) / np.sqrt(2)) / np.sqrt(no / 2)            # should be N(0,1)
    N = z.size
    assert abs(z.mean()) < 5 / np.sqrt(N)
    assert abs(z.var() - 1) < 5 * np.sqrt(2 / N)
    assert abs((z ** 4).mean() - 3) < 5 * np.sqrt(96 / N)
    assert abs(np.mean(z[:, 0::2] * z[:, 1::2])) < 5 / np.sqrt(N / 2)  # real / imaginary parts uncorrelated
    assert abs(np.mean(np.abs(z) > 3) - 0.0026998) < 5 * np.sqrt(0.0027 / N)
    # counter-based stream: pure function of (seed, offset + b, i), independent of the launch geometry
    u2, _, lg2 = dk.awgn_frontend(tables, B // 2, no, seed=99, offset=5 + B // 2)
    assert torch.equal(lg2, lg[B // 2:]) and torch.equal(u2, u[B // 2:])
    _, _, lg3 = dk.awgn_frontend(tables, 64, no, seed=100, offset=5)
    assert not torch.equal(lg3, lg[:64])
    # Mapper/AWGN/Demapper-only entry point reproduces the same noise for the same codewords
    cf = torch.from_numpy(cb.astype(np.float32)).to(dev)
    if n >= 4:
        assert torch.equal(dk.qpsk_awgn_llr(cf, no, seed=99, offset=5), lg)


def test_error_counters_match_numpy():
    torch, dk, po, co, dev = _env()
    rng = np.random.default_rng(3)
    for (B, k) in ((1, 1), (1000, 32), (777, 512), (50, 1000)):
        a = rng.integers(0, 2, size=(B, k)).astype(np.float32)
        b = a.copy()
        flip = rng.random((B, k)) < 0.01
        b[flip] = 1 - b[flip]
        cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        dk.count_errors_f32(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), cnt)
        assert cnt.cpu().tolist() == [po.count_errors(a, b), po.count_block_errors(a, b)]
    n = 256
    a = rng.integers(0, 2, size=(999, n)).astype(np.uint8)
    b = a ^ (rng.random((999, n)) < 0.003)
    mask = rng.integers(0, 2, size=n).astype(np.uint8)
    cnt = torch.zeros(2, dtype=torch.int64, device=dev)
    to = lambda x: torch.from_numpy(pack_words(x).view(np.int32)).to(dev)
    dk.count_errors_packed(to(a), to(b), to(mask[None])[0], n, cnt)
    d = (a != b) & (mask[None] != 0)
    assert cnt.cpu().tolist() == [int(d.sum()), int(d.any(1).sum())]
    from my_sn.sim import count_errors, count_block_errors
    x = torch.from_numpy(a[:, :7].astype(np.float32)).to(dev); y = torch.from_numpy(b[:, :7].astype(np.float32)).to(dev)
    assert int(count_errors(x, y)) == int((a[:, :7] != b[:, :7]).sum())
    assert int(count_block_errors(x, y)) == int((a[:, :7] != b[:, :7]).any(1).sum())


def test_pack_unpack_roundtrip():
    torch, dk, po, co, dev = _env()
    rng = np.random.default_rng(4)
    for n in (8, 32, 96, 1024):
        x = rng.integers(0, 2, size=(257, n)).astype(np.float32)
        p = dk.pack_bits(torch.from_numpy(x).to(dev))
        assert np.array_equal(unpack_words(p.cpu().numpy(), n), x.astype(np.uint8))
        pos = torch.arange(n, dtype=torch.int32, device=dev)
        assert np.array_equal(dk.unpack_info(p, pos, n).cpu().numpy(), x)


@pytest.mark.parametrize("name", golden_names("sclcrc_"))
def test_crc_aided_scl_matches_composed_reference(name):
    torch, dk, po, co, dev = _env()
    from my_sn.fec.polar.dec import SCL_Dec
    d = golden(name)
    n = d["logits"].shape[1]
    dec = SCL_Dec(d["frozen_pos"], n, list_size=8, crc_degree=str(d["crc_degree"]), cn_type="minsum")
    out = dec(torch.from_numpy(d["logits"]).to(dev)).cpu().numpy().astype(np.uint8)
    rb = d["robust"]
    assert np.array_equal(out[rb], d["u_sel"][rb])
    assert dec.k_crc == po.CRC_COEFFS[str(d["crc_degree"])][0]


def test_crc_aided_scl_matches_oracle_random_and_beats_plain_scl():
    torch, dk, po, co, dev = _env()
    from my_sn.fec.polar.dec import SCL_Dec
    from polar.polar_scl import SCL_Dec as PlainSCL
    n, k, L, deg = 128, 64, 8, "CRC11"
    fp = np.asarray(golden("frozen_sets")["g5_128_64"])
    rng = np.random.default_rng(11)
    B = 3000
    payload = rng.integers(0, 2, size=(B, k - 11)).astype(np.uint8)
    bits = po.crc_encode(payload, deg)
    c = po.encode(bits, fp, n)
    no = po.ebnodb2no(2.0, 2, k / n)
    y = (1 - 2.0 * c) / np.sqrt(2) + np.sqrt(no / 2) * rng.standard_normal((B, n))
    logits = (-2 * np.sqrt(2) * y / no).astype(np.float32)
    u_list, pm = co.scl_decode_full(logits, po.frozen_vec(fp, n), L)
    sel, idx = po.scl_crc_select(u_list, pm, fp, n, deg)
    u_b, pm_b = po.scl_decode_full(logits[:600], po.frozen_vec(fp, n), L, use_log1p=True)   # conditioning probe (SURVEY 8c)
    sel_b, _ = po.scl_crc_select(u_b, pm_b, fp, n, deg)
    x = torch.from_numpy(logits).to(dev)
    got = SCL_Dec(fp, n, L, crc_degree=deg, cn_type="minsum")(x).cpu().numpy()
    diff = np.any(got != sel, axis=1)
    probe = np.any(sel_b != sel[:600], axis=1)
    # decisions agree everywhere except (at most) on ill-conditioned codewords, whose rate the two oracle variants bound
    assert diff.mean() <= max(3 * probe.mean(), 2e-3), (diff.mean(), probe.mean())
    assert not diff[:600][~probe].any() or diff.mean() < 2e-3
    plain = PlainSCL(fp, n, L)(x).cpu().numpy()
    bler_aided = np.any(got != bits, axis=1).mean()
    bler_plain = np.any(plain != bits, axis=1).mean()
    assert (idx != 0).sum() > 0 and bler_aided < bler_plain


def test_link_model_and_sim_ber_inside_oracle_confidence_interval():
    """README configuration (k=32, n=64) on the GPU: SC and SCL-8 BLER/BER curves vs the oracle on
    independent noise, 6-sigma binomial bands (both estimates are Monte-Carlo)."""
    torch, dk, po, co, dev = _env()
    from polar.froze import get_Kern_frozen_bits
    from polar.enc import PolarEncoder
    from polar.polar_sc import SC_Dec
    from polar.polar_scl import SCL_Dec
    from z_sys_model.awgn_model import System_AWGN_model
    from my_sn.plotting import PlotBER
    from d_kernels import F2
    n, k, bs = 64, 32, 40000
    fp = golden("frozen_sets")["rm_64_32"]
    ebnos = np.arange(0, 5, 1.0)
    rng = np.random.default_rng(77)
    for name, make, L in (("sc", lambda: SC_Dec(fp, n), 0), ("scl", lambda: SCL_Dec(fp, n, 8), 8)):
        torch.manual_seed(42)
        model = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make())
        plot = PlotBER("t")
        ber, bler = plot.simulate(model, ebnos, batch_size=bs, max_mc_iter=1, add_bler=True, verbose=False, target_block_errs=10 ** 9)
        assert len(plot.ber) == 2 and plot.legend[1].endswith("(BLER)")
        for i, e in enumerate(ebnos):
            u, logits = awgn_logits(rng, n, k, fp, bs, float(e))
            if L == 0:
                hat = co.sc_decode_full(logits, po.frozen_vec(fp, n))[:, po.info_positions(fp, n)]
            else:
                hat = co.scl_decode_full(logits, po.frozen_vec(fp, n), L)[0][:, 0][:, po.info_positions(fp, n)]
            p_ref = np.any(hat != u, axis=1).mean()
            p = float(bler[i])
            band = 6 * np.sqrt(max(p_ref, 1e-4) * (1 - p_ref) / bs * 2) + 1e-4
            assert abs(p - p_ref) < band, (name, e, p, p_ref)
            b_ref = (hat != u).mean()
            assert abs(float(ber[i]) - b_ref) < 6 * np.sqrt(max(b_ref, 1e-4) / bs * 2) + 1e-4, (name, e)
    # README KAT curve (bs=100): the GPU curve must also be compatible with the published points
    kat = golden("readme_kat")
    torch.manual_seed(42)
    model = System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n))
    from my_sn.sim import sim_ber
    ber, bler = sim_ber(model, kat["ebno_dbs"], 20000, 1, verbose=False, early_stop=False)
    for p_pub, p in zip(kat["sc_bler"], bler.numpy()):
        assert abs(p_pub - p) < 5 * np.sqrt(max(p, 1e-3) * (1 - p) / 100) + 0.02
    # layer-by-layer composition (fused=False) gives the same statistics
    m2 = System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n), fused=False)
    b, bh = m2(20000, 2.0)
    p2 = float((b != bh).any(-1).float().mean())
    assert abs(p2 - float(bler[4])) < 6 * np.sqrt(p2 * (1 - p2) / 20000 * 2)
    c, _ = System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n), cw_estimates=True)(16, 2.0)
    assert c.shape == (16, n)


def test_my_sn_encoder_and_parity_check():
    torch, dk, po, co, dev = _env()
    from my_sn.fec.polar.enc import PolarEncoder
    fp = golden("frozen_sets")["rm_256_128"]
    enc = PolarEncoder(fp, 256)
    u = torch.randint(0, 2, (300, 128), device=dev, dtype=torch.float32)
    c = enc(u)
    assert np.array_equal(c.cpu().numpy().astype(np.uint8), po.encode(u.cpu().numpy(), fp, 256))
    assert enc.check_parity(c)
    c[3, 17] = 1 - c[3, 17]
    assert not enc.check_parity(c)
    with pytest.raises(AssertionError):
        enc(torch.zeros(2, 100, device=dev))


@pytest.mark.parametrize("n,B,chunk_mb", [(1024, 5000, 1), (64, 100000, 1), (2048, 700, 128)])
def test_host_buffer_entry_points_match_device_path(n, B, chunk_mb, monkeypatch):
    torch, dk, po, co, dev = _env()
    set_opt("POLAR_HOST_CHUNK_MB", str(chunk_mb))     # several chunks -> exercises the 2-stream pipeline
    k = n // 2
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    _, logits = awgn_logits(np.random.default_rng(n), n, k, fp, B, 3.0)
    _, want = dk.sc_decode(torch.from_numpy(logits).to(dev), tables, want_info=False, want_packed=True)
    h_in = torch.from_numpy(logits).pin_memory()
    h_out = torch.empty((B, dk.words(n)), dtype=torch.int32).pin_memory()
    dk.check(dk.lib().polar_sc_decode_host(h_in.data_ptr(), tables.mask_np.ctypes.data, n, B, h_out.data_ptr(), 0))
    assert torch.equal(h_out, want.cpu())
    Bs = min(B, 600)
    res = dk.scl_decode(torch.from_numpy(logits[:Bs]).to(dev), tables, 4, want_packed=True, want_pm=True, want_info=False)
    h_best = torch.empty((Bs, dk.words(n)), dtype=torch.int32)
    h_pm = torch.empty((Bs, 4), dtype=torch.float64)
    pageable = torch.from_numpy(logits[:Bs].copy())              # pageable memory must work too
    dk.check(dk.lib().polar_scl_decode_host(pageable.data_ptr(), tables.mask_np.ctypes.data, n, 4, Bs, h_best.data_ptr(),
                                            h_pm.data_ptr(), None, 0, 0))
    assert torch.equal(h_best, res["u_packed"].cpu()) and torch.equal(h_pm, res["pm"].cpu())


@pytest.mark.parametrize("chunk_mb", [1, 128])
def test_module_cpu_tensor_path_equals_device_path(chunk_mb):
    """VERDICT r01 #5: SC_Dec / SCL_Dec.forward on a CPU tensor go through polar_{sc,scl}_decode_host_f32 (chunked H2D /
    decode / D2H on two streams, the [B,k] fp32 API tensor straight into page-locked host memory).  Same bits as the
    device-tensor path for page-locked, pageable, non-contiguous and fp64 inputs; CRC-aided selection applies its 30 k
    penalty on the host path too (the packed legacy entry point derives k from the mask)."""
    torch, dk, po, co, dev = _env()
    from polar.polar_sc import SC_Dec
    from polar.polar_scl import SCL_Dec
    from my_sn.fec.polar.dec import SCL_Dec as SclCrc
    from my_sn.fec.crc import CRCEncoder
    set_opt("POLAR_HOST_CHUNK_MB", chunk_mb)
    n, k, B, L = 1024, 512, 3000, 8
    fp = golden("frozen_sets")["rm_1024_512"]
    tables = dk.code_tables(fp, n, dev)
    chk = CRCEncoder("CRC11", k)
    gen = CRCEncoder("CRC11", k - chk.crc_length)
    payload = torch.randint(0, 2, (B, k - gen.crc_length), device=dev, dtype=torch.float32)
    x = dk.qpsk_awgn_llr(dk.encode_f32(gen(payload), tables), po.ebnodb2no(3.0, 2, k / n), 5)
    pinned = torch.empty((B, n), dtype=torch.float32, pin_memory=True); pinned.copy_(x)
    pageable = x.cpu()
    sc = SC_Dec(fp, n)
    want = sc(x).cpu()
    for inp in (pinned, pageable, pageable.double(), pageable.reshape(30, 100, n), torch.cat([pageable, pageable], 1)[:, n:]):
        got = sc(inp)
        assert got.device.type == "cpu" and got.dtype == torch.float32 and torch.equal(got.reshape(B, k), want)
    scl = SCL_Dec(fp, n, L)
    want = scl(x).cpu(); pm = scl.msg_pm.cpu()
    assert torch.equal(scl(pageable), want) and torch.equal(scl.msg_pm, pm) and torch.equal(scl(pinned), want)
    crc = SclCrc(fp, n, L, crc_degree="CRC11", cn_type="minsum")
    want_crc = crc(x).cpu()
    assert not torch.equal(want_crc, want)                       # the CRC picks another candidate on some codewords
    assert torch.equal(crc(pinned), want_crc) and torch.equal(crc(pageable), want_crc)
    # legacy packed entry point (no k argument): same selection as the device call that is told k
    rows = chk.syndrome_rows(tables.info_pos_np, n)
    h_best = torch.empty((B, n // 32), dtype=torch.int32, pin_memory=True)
    dk.check(dk.lib().polar_scl_decode_host(pinned.data_ptr(), tables.mask_np.ctypes.data, n, L, B, h_best.data_ptr(), None,
                                            rows.ctypes.data, chk.crc_length, 0))
    assert torch.equal(dk.unpack_info(h_best.to(dev), tables.info_pos, n).cpu(), want_crc)
    # the device C ABI refuses a CRC-aided call that does not say k (its penalty would silently be 0)
    rows_d = torch.from_numpy(rows.view(np.int32).copy()).to(dev)
    best = torch.empty((B, n // 32), dtype=torch.int32, device=dev)
    need = int(dk.lib().polar_scl_workspace_bytes(n, L, B))
    ws = torch.empty(need + 256, dtype=torch.uint8, device=dev)
    wp = (ws.data_ptr() + 255) // 256 * 256
    rc = dk.lib().polar_scl_decode(dk.ptr(x), dk.ptr(tables.frozen_mask), n, L, B, dk.ptr(best), None, None, 0, None, None,
                                   dk.ptr(rows_d), chk.crc_length, wp, need, dk.stream_ptr(dev))
    assert rc == dk.POLAR_EINVAL


def test_full_size_properties_sc():
    """BASELINE configs[1] size (n=1024, k=512, 2^20 codewords): size-independent properties.
    (a) noiseless codewords decode to the transmitted bits; (b) decisions do not depend on how the batch is
    split across launches; (c) the kernel is deterministic; (d) BLER sits in the oracle's confidence band."""
    torch, dk, po, co, dev = _env()
    n, k, B = 1024, 512, 1 << 20
    fp = golden("frozen_sets")["rm_1024_512"]
    tables = dk.code_tables(fp, n, dev)
    no = po.ebnodb2no(4.0, 2, k / n)
    u, c, lg = dk.awgn_frontend(tables, B, no, seed=5, want_codeword=True)
    _, hat = dk.sc_decode(lg, tables, want_info=False, want_packed=True)
    _, hat2 = dk.sc_decode(lg, tables, want_info=False, want_packed=True)
    assert torch.equal(hat, hat2)
    parts = torch.cat([dk.sc_decode(lg[a:b], tables, want_info=False, want_packed=True)[1]
                       for a, b in ((0, 7), (7, 100003), (100003, B))])
    assert torch.equal(parts, hat)
    cnt = torch.zeros(2, dtype=torch.int64, device=dev)
    dk.count_errors_packed(u, hat, tables.info_mask, n, cnt)
    bler = cnt[1].item() / B
    ref_u, ref_lg = awgn_logits(np.random.default_rng(8), n, k, fp, 20000, 4.0)
    ref_hat = co.sc_decode_full(ref_lg, po.frozen_vec(fp, n))[:, po.info_positions(fp, n)]
    p_ref = np.any(ref_hat != ref_u, axis=1).mean()
    assert abs(bler - p_ref) < 6 * np.sqrt(p_ref * (1 - p_ref) / 20000)
    # noiseless: logits = -/+ big for bit 0/1
    cb = unpack_words(c[:4096].cpu().numpy(), n).astype(np.float32)
    clean = torch.from_numpy((2 * cb - 1) * 8.0).to(dev)
    _, h3 = dk.sc_decode(clean, tables, want_info=False, want_packed=True)
    assert torch.equal(h3, u[:4096])
    # bit-exact vs the oracle on a slice of the full-size batch
    sl = slice(B - 3000, B)
    assert np.array_equal(unpack_words(hat[sl].cpu().numpy(), n), co.sc_decode_full(lg[sl].cpu().numpy(), po.frozen_vec(fp, n)))


@pytest.mark.parametrize("dec_kind", ["sc", "scl4", "scl8_crc"])
def test_on_device_monte_carlo_loop_equals_host_loop(dec_kind):
    """SURVEY 8(f) N1: sim_ber_device (stop rules evaluated by polar_mc_control_group on the GPU, iterations queued ahead)
    must reproduce the host loop counter for counter -- same seed, same number of counted iterations, same status."""
    torch, dk, po, co, dev = _env()
    from polar.enc import PolarEncoder
    from polar.polar_sc import SC_Dec
    from polar.polar_scl import SCL_Dec
    from my_sn.fec.polar.dec import SCL_Dec as SCL_CRC
    from z_sys_model.awgn_model import System_AWGN_model
    from my_sn.sim import sim_ber, sim_ber_device
    n, k, bs = 128, 64, 3000
    fp = po.rm_frozen_pos(n, n - k)
    make = {"sc": lambda: SC_Dec(fp, n), "scl4": lambda: SCL_Dec(fp, n, 4),
            "scl8_crc": lambda: SCL_CRC(fp, n, 8, crc_degree="CRC6")}[dec_kind]
    ebnos = np.array([1.0, 2.5, 4.0, 5.5, 9.0, 10.0], dtype=np.float32)
    for kw in (dict(max_mc_iter=7, target_block_errs=500), dict(max_mc_iter=5, target_bit_errs=2000),
               dict(max_mc_iter=3), dict(max_mc_iter=1, target_block_errs=1)):
        host = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make(), seed=99)
        devm = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make(), seed=99)
        ber_h, bler_h = sim_ber(host, ebnos, bs, verbose=False, on_device=False, **kw)
        ber_d, bler_d, cnt, status, iters = sim_ber_device(devm, ebnos, bs, verbose=False, return_counters=True, **kw)
        assert torch.equal(ber_h, ber_d) and torch.equal(bler_h, bler_d), (dec_kind, kw)
        assert host._offset == devm._offset                       # same number of counted iterations
        assert (iters <= kw["max_mc_iter"]).all()
        # status codes follow sim.py:63-66 / 107-133
        first = int(status[0])
        assert first in (1, 3, 4)
        if "target_block_errs" in kw and cnt[0, 1] >= kw["target_block_errs"]:
            assert first == 4
        if "target_bit_errs" in kw and cnt[0, 0] >= kw["target_bit_errs"]:
            assert first == 3
        # early stop: the sweep ends at the first error-free point, later points stay "not simulated"
        zero = np.nonzero((cnt[:, 1] == 0) & (cnt[:, 3] > 0))[0]
        if len(zero):
            assert status[zero[0]] == 2 and (cnt[zero[0] + 1:] == 0).all()
    # sim_ber routes to the device loop by default and PlotBER.simulate passes the switch through
    a = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make(), seed=5)
    b = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make(), seed=5)
    from my_sn.plotting import PlotBER
    r1 = PlotBER("a").simulate(a, ebnos[:3], bs, max_mc_iter=2, verbose=False)
    r2 = PlotBER("b").simulate(b, ebnos[:3], bs, max_mc_iter=2, verbose=False, on_device=False)
    assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1])


def test_device_loop_lookahead_and_bec_model():
    """(a) A sweep whose points stop after one iteration (configs[3] regime) wastes at most one look-ahead iteration in
    total (StopPredictor), with results identical to the loop without look-ahead.  (b) ADVICE r01: System_BEC_model goes
    through sim_ber on both paths (its own `device_frontend` hook: erasures, not AWGN) with identical counters."""
    torch, dk, po, co, dev = _env()
    from polar.enc import PolarEncoder
    from polar.polar_sc import SC_Dec
    from z_sys_model.awgn_model import System_AWGN_model
    from z_sys_model.bec_model import System_BEC_model
    from my_sn.sim import sim_ber, sim_ber_device
    n, k, bs = 256, 128, 4096
    fp = po.rm_frozen_pos(n, n - k)
    ebnos = np.array([0.0, 0.5, 1.0, 1.5, 2.0], dtype=np.float32)           # BLER >> 100 / 4096 everywhere
    mk = lambda: System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n), seed=17)
    st_a, st_b = {}, {}
    a = sim_ber_device(mk(), ebnos, bs, 16, target_block_errs=100, verbose=False, return_counters=True, stats=st_a)
    b = sim_ber_device(mk(), ebnos, bs, 16, target_block_errs=100, verbose=False, return_counters=True, stats=st_b, lookahead=False)
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4])
    assert st_b["queued"] == st_b["counted"] == len(ebnos)
    assert st_a["counted"] == len(ebnos) and st_a["queued"] <= len(ebnos) + 1, st_a
    # long points: look-ahead stays on (one discarded iteration per point at most)
    st_c = {}
    sim_ber_device(mk(), np.array([4.0, 4.5], dtype=np.float32), 512, 12, target_block_errs=10 ** 6, verbose=False, stats=st_c)
    assert st_c["counted"] == 24 and st_c["queued"] == 24
    from types import SimpleNamespace
    pes = np.array([0.5, 0.4, 0.3], dtype=np.float32)
    mb = lambda: System_BEC_model(SimpleNamespace(n=n, k=k), PolarEncoder(fp, n, None), SC_Dec(fp, n), seed=23)
    r_dev = sim_ber(mb(), pes, 2000, 3, target_block_errs=50, verbose=False)
    r_host = sim_ber(mb(), pes, 2000, 3, target_block_errs=50, verbose=False, on_device=False)
    assert torch.equal(r_dev[0], r_host[0]) and torch.equal(r_dev[1], r_host[1])
    assert 0.0 < float(r_dev[1][2]) < float(r_dev[1][0]) <= 1.0


def test_on_device_loop_with_process_group_of_one():
    """The sharded path (stream-ordered NCCL all-reduce of the counters before polar_mc_control_group) with world size 1."""
    torch, dk, po, co, dev = _env()
    import torch.distributed as dist
    from polar.enc import PolarEncoder
    from polar.polar_sc import SC_Dec
    from z_sys_model.awgn_model import System_AWGN_model
    from my_sn.sim import sim_ber_device
    n, k, bs = 256, 128, 2000
    fp = po.rm_frozen_pos(n, n - k)
    ebnos = np.array([2.0, 4.0], dtype=np.float32)
    ref = sim_ber_device(System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n), seed=3), ebnos, bs, 3,
                         target_block_errs=100, verbose=False, return_counters=True)
    # an in-process store: a group of one needs no TCP rendezvous, so no port that another job on the host could hold
    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1)
    try:
        got = sim_ber_device(System_AWGN_model(n, k, PolarEncoder(fp, n, None), SC_Dec(fp, n), seed=3), ebnos, bs, 3,
                             target_block_errs=100, verbose=False, return_counters=True)
    finally:
        dist.destroy_process_group()
    assert np.array_equal(ref[2], got[2]) and np.array_equal(ref[3], got[3])


def test_full_size_properties_scl_configs():
    """BASELINE configs[2] (SCL L=8, n=1024, CRC11, 2^18 codewords) and configs[3] (SCL L=32, n=2048, k=1024) at full
    list size: (a) split-invariance and determinism of the whole batch; (b) noiseless codewords decode to the transmitted
    bits with path metric 0; (c) the list decoder is never worse than SC on the same noise and CRC-aided selection is
    never worse than plain selection; (d) a slice of the full batch is bit-exact against the oracle."""
    torch, dk, po, co, dev = _env()
    from my_sn.fec.crc import CRCEncoder
    # ---- configs[2]
    n, k, B, L = 1024, 512, 1 << 18, 8
    fp = golden("frozen_sets")["rm_1024_512"]
    tables = dk.code_tables(fp, n, dev)
    chk = CRCEncoder("CRC11", k)
    gen = CRCEncoder("CRC11", k - chk.crc_length)
    rows = torch.from_numpy(chk.syndrome_rows(tables.info_pos_np, n).view(np.int32).copy()).to(dev)
    payload = torch.randint(0, 2, (B, k - gen.crc_length), device=dev, dtype=torch.float32)
    bits = gen(payload)
    cw = dk.encode_f32(bits, tables)
    lg = dk.qpsk_awgn_llr(cw, po.ebnodb2no(3.5, 2, k / n), 777)
    full = torch.zeros((B, n), dtype=torch.float32, device=dev)
    full[:, tables.info_pos.long()] = bits
    tx = dk.pack_bits(full)
    aided = dk.scl_decode(lg, tables, L, crc_rows=rows, crc_len=chk.crc_length, want_info=False, want_packed=True)["u_packed"]
    again = dk.scl_decode(lg, tables, L, crc_rows=rows, crc_len=chk.crc_length, want_info=False, want_packed=True)["u_packed"]
    assert torch.equal(aided, again)
    parts = torch.cat([dk.scl_decode(lg[a:b], tables, L, crc_rows=rows, crc_len=chk.crc_length, want_info=False,
                                     want_packed=True)["u_packed"] for a, b in ((0, 3), (3, 70001), (70001, B))])
    assert torch.equal(parts, aided)
    plain = dk.scl_decode(lg, tables, L, want_info=False, want_packed=True)["u_packed"]
    _, sc = dk.sc_decode(lg, tables, want_info=False, want_packed=True)

    def bler(hat):
        cnt = torch.zeros(2, dtype=torch.int64, device=dev)
        dk.count_errors_packed(tx, hat, tables.info_mask, n, cnt)
        return cnt[1].item() / B
    b_aided, b_plain, b_sc = bler(aided), bler(plain), bler(sc)
    assert b_aided <= b_plain + 1e-3 and b_plain <= b_sc + 1e-3 and b_aided < 0.9 * b_sc, (b_aided, b_plain, b_sc)
    sl = slice(B - 48, B)
    u_ref, pm_ref = co.scl_decode_full(lg[sl].cpu().numpy(), po.frozen_vec(fp, n), L)
    got = dk.scl_decode(lg[sl], tables, L, want_info=False, want_packed=True, want_pm=True)
    assert np.array_equal(unpack_words(got["u_packed"].cpu().numpy(), n), u_ref[:, 0])
    assert np.allclose(got["pm"].cpu().numpy()[:, 0], pm_ref[:, 0], rtol=1e-5, atol=1e-9)
    assert torch.equal(got["u_packed"], plain[sl])
    # ---- configs[3]: L = 32, n = 2048
    n, k, B, L = 2048, 1024, 1 << 13, 32
    fp = golden("frozen_sets")["rm_2048_1024"]
    tables = dk.code_tables(fp, n, dev)
    u, c, lg = dk.awgn_frontend(tables, B, po.ebnodb2no(3.0, 2, k / n), seed=11, want_codeword=True)
    res = dk.scl_decode(lg, tables, L, want_info=False, want_packed=True, want_pm=True)
    _, sc = dk.sc_decode(lg, tables, want_info=False, want_packed=True)
    cnt = torch.zeros(2, dtype=torch.int64, device=dev); cnt2 = torch.zeros(2, dtype=torch.int64, device=dev)
    dk.count_errors_packed(u, res["u_packed"], tables.info_mask, n, cnt)
    dk.count_errors_packed(u, sc, tables.info_mask, n, cnt2)
    assert cnt[1].item() <= cnt2[1].item()
    pm = res["pm"].cpu().numpy()
    assert (np.diff(pm, axis=1) >= 0).all()                         # list is sorted by path metric
    cb = unpack_words(c[:512].cpu().numpy(), n).astype(np.float32)
    clean = torch.from_numpy((2 * cb - 1) * 40.0).to(dev)            # |LLR| > 30: clipped, penalty log(1+e^-30) per leaf
    r2 = dk.scl_decode(clean, tables, L, want_info=False, want_packed=True, want_pm=True)
    assert torch.equal(r2["u_packed"], u[:512])
    assert np.allclose(r2["pm"].cpu().numpy()[:, 0], n * np.log1p(np.exp(-30.0)), rtol=1e-9)
    u_ref, pm_ref = co.scl_decode_full(lg[:6].cpu().numpy(), po.frozen_vec(fp, n), L)
    assert np.array_equal(unpack_words(res["u_packed"][:6].cpu().numpy(), n), u_ref[:, 0])


def test_5g_encoder_decoder_wrappers():
    """SURVEY 8f N3 on the GPU: Polar5GEncoder output bit-exact with the reference's codewords (CRC + polar transform +
    one gather), polar_rate_recover_f32 exact against the reference's de-rate-matched logits, and the encode -> AWGN ->
    Polar5GDecoder loop (SC, CRC-aided SCL, crc status) recovering the payload."""
    torch, dk, po, co, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    g = golden("nr5g")
    for k, n in g["cfgs"]:
        key = "%d_%d" % (k, n)
        enc = Polar5GEncoder(int(k), int(n))
        c = enc(torch.from_numpy(g["u_" + key].astype(np.float32)).cuda())
        assert c.shape == (6, n) and np.array_equal(c.cpu().numpy().astype(np.uint8), g["c_" + key]), key
        dec = Polar5GDecoder(enc, dec_type="SC")
        dem = dec.rate_recover(torch.from_numpy(g["llr_" + key]).cuda())
        assert np.array_equal(dem.cpu().numpy(), g["dem_" + key]), key
    torch.manual_seed(3)
    for (k, n, ebno) in ((64, 128, 5.0), (100, 300, 3.0), (200, 256, 6.5), (300, 1088, 2.0)):
        enc = Polar5GEncoder(k, n)
        B = 3000
        u = torch.randint(0, 2, (B, k), device=dev, dtype=torch.float32)
        c = enc(u)
        no = po.ebnodb2no(ebno, 2, k / n)
        llr = dk.qpsk_awgn_llr(c.contiguous(), no, 99) if n % 2 == 0 else None
        assert llr is not None
        res = {}
        for kind in ("SC", "SCL"):
            dec = Polar5GDecoder(enc, dec_type=kind, list_size=8)
            hat = dec(llr)
            assert hat.shape == (B, k)
            res[kind] = (hat != u).any(-1).float().mean().item()
        assert res["SCL"] <= res["SC"] + 0.01 and res["SCL"] < 0.2, (k, n, res)
        hat, ok = Polar5GDecoder(enc, dec_type="SCL", list_size=8, return_crc_status=True)(llr)
        good = ~(hat != u).any(-1)
        assert ok.shape == (B,) and (ok.bool() | ~good).float().mean().item() > 0.999      # decoded correctly => CRC holds
        # noiseless: exact recovery through rate recovery for every scheme
        clean = (2 * c - 1) * 10.0
        assert torch.equal(Polar5GDecoder(enc, dec_type="SCL")(clean), u)
    with pytest.raises(Exception):
        Polar5GEncoder(30, 108, channel_type="downlink")(torch.zeros(2, 30).cuda())


def test_bec_channel_and_link_model():
    """SURVEY 8f N4 (channel half): polar_bec_frontend / polar_bec_llr statistics, the BinaryErasureChannel layer in both
    output modes, and System_BEC_model's BLER inside the confidence band of the oracle SC decoder on independent erasures."""
    torch, dk, po, co, dev = _env()
    from types import SimpleNamespace
    from polar.enc import PolarEncoder
    from polar.polar_sc import SC_Dec
    from z_sys_model.bec_model import System_BEC_model
    from my_sn.trans.channel.discrete_channel import BinaryErasureChannel
    n, k, B, pe = 256, 128, 40000, 0.35
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    u, c, llr = dk.bec_frontend(tables, B, pe, seed=7, want_codeword=True)
    x = llr.cpu().numpy()
    cb = unpack_words(c.cpu().numpy(), n)
    er = x == 0
    assert abs(er.mean() - pe) < 5 * np.sqrt(pe * (1 - pe) / x.size)
    assert np.array_equal(x[~er], np.where(cb[~er] == 1, 100.0, -100.0).astype(np.float32))
    assert abs(er[:, 0].mean() - pe) < 6 * np.sqrt(pe * (1 - pe) / B) and abs(er[:, n - 1].mean() - pe) < 6 * np.sqrt(pe * (1 - pe) / B)
    u2, _, llr2 = dk.bec_frontend(tables, B, pe, seed=7)
    assert torch.equal(llr, llr2) and torch.equal(u, u2)                      # pure function of (seed, offset)
    # layer API
    ch = BinaryErasureChannel(return_llrs=True)
    bits = torch.randint(0, 2, (500, n), device=dev, dtype=torch.float32)
    y = ch([bits, 0.2])
    assert set(np.unique(y.cpu().numpy())) <= {-100.0, 0.0, 100.0} and abs((y == 0).float().mean().item() - 0.2) < 0.01
    assert torch.equal(y[y != 0], torch.where(bits[y != 0] == 1, 100.0, -100.0))
    t = BinaryErasureChannel(return_llrs=False)([bits, 0.5])
    assert set(np.unique(t.cpu().numpy())) <= {-1.0, 0.0, 1.0} and torch.equal(t[t >= 0], bits[t >= 0])
    tb = BinaryErasureChannel(return_llrs=False, bipolar_input=True)([2 * bits - 1, 0.5])
    assert set(np.unique(tb.cpu().numpy())) <= {-1.0, 0.0, 1.0} and torch.equal(tb[tb != 0], (2 * bits - 1)[tb != 0])
    with pytest.raises(AssertionError):
        BinaryErasureChannel(return_llrs=True)([bits + 2, 0.1])
    # link model vs oracle
    cfg = SimpleNamespace(n=n, k=k)
    model = System_BEC_model(cfg, PolarEncoder(fp, n, None), SC_Dec(fp, n), seed=5)
    b, bh = model(B, pe)
    bler = (b != bh).any(-1).float().mean().item()
    rng = np.random.default_rng(3)
    ub = rng.integers(0, 2, (8000, k)).astype(np.uint8)
    cw = po.encode(ub, fp, n)
    lg = np.where(cw == 1, 100.0, -100.0).astype(np.float32)
    lg[rng.random(lg.shape) < pe] = 0.0
    ref = co.sc_decode_full(lg, po.frozen_vec(fp, n))[:, po.info_positions(fp, n)]
    p_ref = np.any(ref != ub, axis=1).mean()
    assert abs(bler - p_ref) < 6 * np.sqrt(max(p_ref, 1e-3) * (1 - p_ref) / 8000)
    m2 = System_BEC_model(cfg, PolarEncoder(fp, n, None), SC_Dec(fp, n), fused=False)
    b2, bh2 = m2(8000, pe)
    assert abs((b2 != bh2).any(-1).float().mean().item() - p_ref) < 8 * np.sqrt(max(p_ref, 1e-3) * (1 - p_ref) / 8000)


def test_mc_control_group_follows_the_sequential_stop_rules():
    """polar_mc_control_group against a plain Python walk of sim.py:79-133 over the same per-iteration counters: items that
    the sequential loop would not have run at their position (wrong point after an early / late stop, anything behind such an
    item, anything after the sweep ended, a group planned for another position) must not count."""
    torch, dk, po, co, dev = _env()
    rng = np.random.default_rng(5)

    def reference(deltas, points, P, q0_expect, sweep0, state0, tb, tk, mx, early):
        st, sw = state0.copy(), sweep0.copy()
        consumed = 0
        if not sw[1] and sw[2] == q0_expect:
            for d, p in zip(deltas, points):
                pc = sw[0]
                if pc >= P or p != pc:
                    break
                st[pc, :4] += d; st[pc, 6] += 1; sw[2] += 1; consumed += 1
                if tb is not None and st[pc, 0] >= tb: st[pc, 5], st[pc, 4] = 3, 1
                elif tk is not None and st[pc, 1] >= tk: st[pc, 5], st[pc, 4] = 4, 1
                elif st[pc, 6] >= mx: st[pc, 5], st[pc, 4] = 1, 1
                if st[pc, 4]:
                    if early and st[pc, 1] == 0:
                        st[pc, 5] = 2; sw[1] = 1
                        break
                    sw[0] = pc + 1
                    if pc + 1 >= P:
                        sw[1] = 1
                        break
        sw[3] += 1; sw[4] = consumed
        return st, sw

    for trial in range(60):
        P = int(rng.integers(1, 6)); mx = int(rng.integers(1, 5))
        tb = None if rng.random() < 0.5 else int(rng.integers(1, 60))
        tk = None if rng.random() < 0.5 else int(rng.integers(1, 12))
        early = bool(rng.random() < 0.7)
        state = torch.zeros((P, 8), dtype=torch.int64, device=dev)
        sweep = torch.zeros(8, dtype=torch.int64, device=dev)
        st_ref, sw_ref = np.zeros((P, 8), dtype=np.int64), np.zeros(8, dtype=np.int64)
        for group in range(6):
            G = int(rng.integers(1, dk.MC_GROUP_MAX + 1))
            lo = int(min(sw_ref[0], P - 1))
            hi = max(min(P, lo + 3) + int(rng.random() < 0.2), lo + 1)
            pts = np.sort(rng.integers(lo, hi, size=G)).tolist()           # plausible and wrong plans
            deltas = np.stack([rng.integers(0, 25, G) * (rng.random(G) < 0.8), rng.integers(0, 4, G) * (rng.random(G) < 0.7),
                               np.full(G, 640), np.full(G, 10)], axis=1).astype(np.int64)
            expect_q = int(sw_ref[2]) if rng.random() < 0.85 else int(sw_ref[2]) + 1
            d_dev = torch.from_numpy(deltas).to(dev)
            dk.mc_control_group(d_dev, pts, state, sweep, expect_q, tb, tk, mx, early)
            st_ref, sw_ref = reference(deltas, pts, P, expect_q, sw_ref, st_ref, tb, tk, mx, early)
            assert np.array_equal(state.cpu().numpy(), st_ref), (trial, group)
            assert np.array_equal(sweep.cpu().numpy(), sw_ref), (trial, group)
            assert not d_dev.any()                                   # the call clears the counters it consumed or ignored
    L = dk.lib()
    st = dk.stream_ptr(dev)
    import ctypes
    one = (ctypes.c_int32 * 1)(0)
    assert L.polar_mc_control_group(None, ctypes.cast(one, ctypes.c_void_p), 1, dk.ptr(state), 1, dk.ptr(sweep), 0, -1, -1, 1, 1, st) == dk.POLAR_EINVAL
    assert L.polar_mc_control_group(dk.ptr(sweep), ctypes.cast(one, ctypes.c_void_p), 33, dk.ptr(state), 1, dk.ptr(sweep), 0, -1, -1, 1, 1, st) == dk.POLAR_EINVAL
    assert L.polar_mc_control_group(dk.ptr(sweep), ctypes.cast(one, ctypes.c_void_p), 1, dk.ptr(state), 1, dk.ptr(sweep), 0, -1, -1, 0, 1, st) == dk.POLAR_EINVAL
