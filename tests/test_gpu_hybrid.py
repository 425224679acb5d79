"""Hybrid SC -> SCL decoding (polar_scl_decode_hybrid, SCL_Dec(use_hybrid_sc=True), Polar5GDecoder(dec_type="hybSCL")).

The result is defined by composition of paths that are already pinned to the reference: for every row, the SC decision
of the same arithmetic if its CRC holds (numpy CRC, oracle.polar_oracle.crc_valid), else the CRC-aided list decision of
the existing full-batch list decoder.  The hybrid must equal that composition bit for bit."""
import numpy as np
import pytest

from oracle.polar_oracle import CRC_COEFFS

CRC_LEN = {deg: c[0] for deg, c in CRC_COEFFS.items()}
MINSUM, BOXPLUS, PRUNED = 0, 1, 2


def _env():
    import torch
    import d_kernels as dk
    from oracle import polar_oracle as po
    return torch, dk, po, torch.device("cuda", 0)


def _code(dk, po, n, k, deg, dev):
    import torch
    from my_sn.fec.crc import CRCEncoder
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    rows = torch.from_numpy(CRCEncoder(deg, k).syndrome_rows(tables.info_pos_np, n).view(np.int32).copy()).to(dev)
    return fp, tables, rows


def _crc_logits(torch, dk, po, tables, deg, B, ebno, seed):
    """Logits of B codewords whose k information bits carry a valid CRC, through the device QPSK/AWGN channel."""
    from my_sn.fec.crc import CRCEncoder
    k = tables.k
    g = torch.Generator(device=tables.dev).manual_seed(seed)
    payload = torch.randint(0, 2, (B, k - CRC_LEN[deg]), generator=g, device=tables.dev).float()
    bits = CRCEncoder(deg, k - CRC_LEN[deg])(payload)
    cw = dk.encode_f32(bits, tables)
    return bits, dk.qpsk_awgn_llr(cw, po.ebnodb2no(ebno, 2, k / tables.n), seed)


def _composition(torch, dk, po, lg, tables, L, rows, deg, mode):
    """SC of the mode's arithmetic, numpy CRC check, full-batch CRC-aided list decode -> (u_info, u_packed, SC passed)."""
    boxplus = mode != MINSUM
    u_sc, p_sc = dk.sc_decode(lg, tables, want_info=True, want_packed=True, boxplus=boxplus)
    full = dk.scl_decode(lg, tables, L, crc_rows=rows, crc_len=CRC_LEN[deg], want_info=True, want_packed=True,
                         boxplus=boxplus, pruned=mode == PRUNED)
    ok = po.crc_valid(u_sc.cpu().numpy().astype(np.uint8), deg)
    okt = torch.from_numpy(ok).to(lg.device)[:, None]
    return torch.where(okt, u_sc, full["u_info"]), torch.where(okt, p_sc, full["u_packed"]), ok


def _hybrid(torch, dk, lg, tables, L, rows, deg, mode, **kw):
    cnt = torch.full((1,), -7, dtype=torch.int32, device=tables.dev)
    res = dk.scl_decode_hybrid(lg, tables, L, rows, CRC_LEN[deg], mode, want_info=True, want_packed=True, n_list_out=cnt, **kw)
    return res["u_info"], res["u_packed"], int(cnt.item())


# (cn_mode, n, k, CRC, L, B, Eb/N0): a covering subset of {min-sum, boxplus, pruned} x codes x L x B x {none, some, all fail}
CASES = [
    (MINSUM, 64, 32, "CRC6", 1, 1, 1.5),
    (BOXPLUS, 64, 32, "CRC6", 32, 3, -3.0),
    (PRUNED, 64, 32, "CRC6", 4, 1001, 1.5),
    (MINSUM, 128, 64, "CRC11", 4, 1001, -3.0),
    (BOXPLUS, 128, 64, "CRC11", 8, 1001, 1.5),
    (PRUNED, 128, 64, "CRC11", 32, 1001, 10.0),
    (MINSUM, 1024, 512, "CRC11", 8, 1 << 16, 4.0),
    (MINSUM, 1024, 512, "CRC11", 8, 1 << 16, 10.0),
    (PRUNED, 1024, 512, "CRC11", 8, 1 << 16, 4.0),
    (BOXPLUS, 1024, 512, "CRC11", 1, 1001, 10.0),
    (MINSUM, 2048, 1024, "CRC24C", 32, 1001, 4.0),
    (PRUNED, 2048, 1024, "CRC24C", 8, 1001, -3.0),
    (BOXPLUS, 2048, 1024, "CRC24C", 4, 3, 10.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,n,k,deg,L,B,ebno", CASES)
def test_hybrid_equals_composition(mode, n, k, deg, L, B, ebno):
    torch, dk, po, dev = _env()
    fp, tables, rows = _code(dk, po, n, k, deg, dev)
    _, lg = _crc_logits(torch, dk, po, tables, deg, B, ebno, seed=n + B + mode)
    want_info, want_packed, ok = _composition(torch, dk, po, lg, tables, L, rows, deg, mode)
    got_info, got_packed, n_list = _hybrid(torch, dk, lg, tables, L, rows, deg, mode)
    assert torch.equal(got_packed, want_packed)
    assert torch.equal(got_info, want_info)
    assert n_list == int((~ok).sum())
    if B >= 1000:                                   # the Eb/N0 points put the failing fraction where they are meant to
        frac = n_list / B
        assert (frac == 0.0) if ebno >= 10 else (frac > 0.95) if ebno <= -3 else (0.0 < frac < 1.0), frac


@pytest.mark.gpu
def test_no_failing_rows_keeps_sc_and_sentinels_are_overwritten():
    torch, dk, po, dev = _env()
    n, k, deg, L, B = 1024, 512, "CRC11", 8, 4099
    fp, tables, rows = _code(dk, po, n, k, deg, dev)
    bits, lg = _crc_logits(torch, dk, po, tables, deg, B, 10.0, seed=3)
    clean = (2 * dk.encode_f32(bits, tables) - 1) * 20.0        # noiseless: SC decodes every row, every CRC holds
    for mode in (MINSUM, PRUNED):
        u_sc, p_sc = dk.sc_decode(clean, tables, want_info=True, want_packed=True, boxplus=mode != MINSUM)
        got_info, got_packed, n_list = _hybrid(torch, dk, clean, tables, L, rows, deg, mode)
        assert n_list == 0 and torch.equal(got_packed, p_sc) and torch.equal(got_info, u_sc) and torch.equal(got_info, bits)
    # failing rows present; outputs pre-filled with sentinels; SC decisions staged in the workspace when no packed output
    _, lg = _crc_logits(torch, dk, po, tables, deg, B, 4.0, seed=4)
    mode = MINSUM
    want_info, want_packed, ok = _composition(torch, dk, po, lg, tables, L, rows, deg, mode)
    assert 0 < (~ok).sum() < B
    need = int(dk.lib().polar_scl_hybrid_workspace_bytes(n, L, B, mode))
    ws = torch.empty(need + 512, dtype=torch.uint8, device=dev)
    wp = (ws.data_ptr() + 255) // 256 * 256
    info = torch.full((B, k), 7.0, device=dev)
    packed = torch.full((B, n // 32), -1, dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    call = lambda p_out, i_out, w, nbytes, crc_len=CRC_LEN[deg], b=B: dk.lib().polar_scl_decode_hybrid(
        dk.ptr(lg), dk.ptr(tables.frozen_mask), n, L, b, dk.ptr(p_out), dk.ptr(i_out), dk.ptr(tables.info_pos), k,
        dk.ptr(rows), crc_len, mode, dk.ptr(cnt), w, nbytes, dk.stream_ptr(dev))
    dk.check(call(None, info, wp, need))
    assert torch.equal(info, want_info) and cnt.item() == int((~ok).sum())
    dk.check(call(packed, None, wp, need))
    assert torch.equal(packed, want_packed)
    # argument checks on the device path
    assert call(packed, info, wp + 8, need) == dk.POLAR_EALIGN
    assert call(packed, info, wp, need - 1) == dk.POLAR_ENOMEM
    assert call(packed, info, wp, need, crc_len=0) == dk.POLAR_EINVAL
    assert call(None, None, wp, need) == dk.POLAR_EINVAL
    before = dk.launch_count()
    assert call(packed, info, wp, need, b=0) == dk.POLAR_OK and dk.launch_count() == before


def test_hybrid_argument_checks_without_gpu():
    import d_kernels as dk
    from my_sn.fec.polar.dec import SCL_Dec
    from oracle import polar_oracle as po
    fp = po.rm_frozen_pos(64, 32)
    with pytest.raises(ValueError, match="crc_degree"):
        SCL_Dec(fp, 64, 8, use_hybrid_sc=True)
    lib = dk.lib()
    dummy = 256
    args = lambda n=64, L=8, B=5, k=32, crc_len=6, mode=0, rows=dummy: (
        dummy, dummy, n, L, B, dummy, None, None, k, rows, crc_len, mode, None, dummy, 1 << 30, None)
    assert lib.polar_scl_decode_hybrid(*args(crc_len=0)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(crc_len=33)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(rows=None)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(k=0)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(k=65)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(mode=3)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(L=3)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(n=8192)) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode_hybrid(*args(B=-1)) == dk.POLAR_EINVAL
    before = lib.polar_launch_count()
    assert lib.polar_scl_decode_hybrid(*args(B=0)) == dk.POLAR_OK and lib.polar_launch_count() == before
    assert lib.polar_scl_hybrid_workspace_bytes(64, 8, 0, 0) == 0 and lib.polar_scl_hybrid_workspace_bytes(64, 8, 5, 3) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("cn_type,use_fast_scl", [("minsum", True), ("boxplus", False), ("boxplus", True)])
def test_module_cpu_and_gpu_tensors_and_packed_path(cn_type, use_fast_scl):
    torch, dk, po, dev = _env()
    from my_sn.fec.polar.dec import SCL_Dec
    n, k, deg, L, B = 256, 128, "CRC11", 8, 3000
    fp, tables, rows = _code(dk, po, n, k, deg, dev)
    mode = MINSUM if cn_type == "minsum" else PRUNED if use_fast_scl else BOXPLUS
    _, lg = _crc_logits(torch, dk, po, tables, deg, B, 3.0, seed=21)
    want_info, want_packed, ok = _composition(torch, dk, po, lg, tables, L, rows, deg, mode)
    dec = SCL_Dec(fp, n, L, crc_degree=deg, use_hybrid_sc=True, use_fast_scl=use_fast_scl, cn_type=cn_type)
    got = dec(lg)
    assert got.is_cuda and torch.equal(got, want_info) and dec.msg_pm is None
    assert int(dec.list_decoded.item()) == int((~ok).sum()) and 0 < int(dec.list_decoded.item()) < B
    got_cpu = dec(lg.cpu().reshape(30, 100, n))
    assert got_cpu.device.type == "cpu" and torch.equal(got_cpu.reshape(B, k), want_info.cpu())
    out = torch.empty((B, n // 32), dtype=torch.int32, device=dev)
    assert dec.decode_packed(lg, tables, out=out) is out and torch.equal(out, want_packed)
    assert torch.equal(dk.unpack_info(out, tables.info_pos, n), got)


@pytest.mark.gpu
def test_5g_decoder_hybrid_equals_rate_recovery_then_composition():
    torch, dk, po, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    torch.manual_seed(5)
    seen_fail = 0
    for (k, n, ebno) in ((64, 128, 2.0), (100, 300, 1.0), (300, 1088, 1.0)):
        enc = Polar5GEncoder(k, n)
        B = 2000
        u = torch.randint(0, 2, (B, k), device=dev, dtype=torch.float32)
        llr = dk.qpsk_awgn_llr(enc(u).contiguous(), po.ebnodb2no(ebno, 2, k / n), 7)
        dec = Polar5GDecoder(enc, dec_type="hybSCL", list_size=8)
        inner = dec._polar_dec
        assert inner._use_hybrid_sc and inner._pruned and inner.list_size == 8
        got = dec(llr)
        deg = enc.enc_crc.crc_degree
        tables = dk.code_tables(inner.frozen_pos, inner.n, dev)
        rows = torch.from_numpy(inner._crc_rows_np.view(np.int32).copy()).to(dev)
        comp, _, ok = _composition(torch, dk, po, dec.rate_recover(llr), tables, 8, rows, deg, PRUNED)
        assert torch.equal(got, comp[:, :-inner.k_crc]), (k, n)
        assert int(inner.list_decoded.item()) == int((~ok).sum())
        seen_fail += int((~ok).sum())
    assert seen_fail > 0


@pytest.mark.gpu
def test_monte_carlo_loops_and_block_error_identity():
    torch, dk, po, dev = _env()
    from polar.enc import PolarEncoder
    from my_sn.fec.polar.dec import SCL_Dec
    from z_sys_model.awgn_model import System_AWGN_model
    from my_sn.sim import sim_ber, sim_ber_device
    n, k, deg, L, bs = 128, 64, "CRC6", 8, 3000
    fp = po.rm_frozen_pos(n, n - k)
    make = lambda: SCL_Dec(fp, n, L, crc_degree=deg, use_hybrid_sc=True)
    ebnos = np.array([1.0, 2.5, 4.0, 5.5, 9.0, 10.0], dtype=np.float32)
    for kw in (dict(max_mc_iter=7, target_block_errs=500), dict(max_mc_iter=5, target_bit_errs=2000),
               dict(max_mc_iter=3), dict(max_mc_iter=1, target_block_errs=1)):
        host = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make(), seed=99)
        devm = System_AWGN_model(n, k, PolarEncoder(fp, n, None), make(), seed=99)
        ber_h, bler_h = sim_ber(host, ebnos, bs, verbose=False, on_device=False, **kw)
        ber_d, bler_d = sim_ber_device(devm, ebnos, bs, verbose=False, return_counters=True, **kw)[:2]
        assert torch.equal(ber_h, ber_d) and torch.equal(bler_h, bler_d), kw
        assert host._offset == devm._offset
    # per row: hybrid = SC where SC passed the CRC, = full CRC-aided SCL elsewhere (boxplus pruned, the default)
    _, tables, rows = _code(dk, po, n, k, deg, dev)
    bits, lg = _crc_logits(torch, dk, po, tables, deg, 20000, 2.0, seed=13)
    full_tx = torch.zeros((bits.shape[0], n), dtype=torch.float32, device=dev)
    full_tx[:, tables.info_pos.long()] = bits
    u_tx = dk.pack_bits(full_tx)
    dec = make()
    hyb = dec.decode_packed(lg, tables)
    _, sc = dk.sc_decode(lg, tables, want_info=False, want_packed=True, boxplus=True)
    full = SCL_Dec(fp, n, L, crc_degree=deg).decode_packed(lg, tables)
    info = tables.info_mask[None]
    err = lambda hat: ((hat ^ u_tx) & info).ne(0).any(1).cpu().numpy()
    passed = po.crc_valid(dk.unpack_info(sc, tables.info_pos, n).cpu().numpy().astype(np.uint8), deg)
    e_h, e_s, e_f = err(hyb), err(sc), err(full)
    assert passed.any() and (~passed).any()
    assert int(e_h.sum()) - int(e_f.sum()) == int(e_s[passed].sum()) - int(e_f[passed].sum())
    assert torch.equal(hyb[torch.from_numpy(~passed).to(dev)], full[torch.from_numpy(~passed).to(dev)])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [MINSUM, PRUNED])
def test_cuda_graph_capture_and_replay(mode):
    torch, dk, po, dev = _env()
    n, k, deg, L, B = 1024, 512, "CRC11", 8, 4096
    fp, tables, rows = _code(dk, po, n, k, deg, dev)
    _, lg1 = _crc_logits(torch, dk, po, tables, deg, B, 1.5, seed=31)
    _, lg2 = _crc_logits(torch, dk, po, tables, deg, B, 2.0, seed=32)
    x = lg1.clone()
    packed = torch.empty((B, n // 32), dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    run = lambda: dk.scl_decode_hybrid(x, tables, L, rows, CRC_LEN[deg], mode, want_info=False, out_packed=packed,
                                       n_list_out=cnt)
    run()                                                    # eager: workspace and kernel attributes in place
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    x.copy_(lg2)
    g.replay()
    torch.cuda.synchronize()
    got, got_cnt = packed.clone(), int(cnt.item())
    want = dk.scl_decode_hybrid(lg2, tables, L, rows, CRC_LEN[deg], mode, want_info=False, want_packed=True,
                                n_list_out=cnt)["u_packed"]
    assert torch.equal(got, want) and got_cnt == int(cnt.item()) and got_cnt > 0
