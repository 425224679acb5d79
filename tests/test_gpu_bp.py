"""Belief-propagation polar decoder (`polar_belief_decode_f32`, my_sn `BP_Dec`, `Polar5GDecoder(dec_type="BP")`).

`bp_decode_full` below is the numpy restatement of the decoder's schedule (csrc/polar_belief.cu); it reuses the SC
oracle's f of each arithmetic.  Under min-sum the kernel equals it bit for bit (soft outputs as values: +0 and -0 are
equal).  Under boxplus the exp / log come from different libraries, so the comparison is statistical: boxplus BP
oscillates on words it fails, where a 1-ulp change of any exp / log result already changes the restatement's own
decision on a large share of them."""
import ctypes

import numpy as np
import pytest

from util import unpack_words

from oracle import polar_oracle as po

NS = [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024]
LLR_MAX = np.float32(po.LLR_MAX)


def _pairs(n, s):
    i = np.arange(n)
    i = i[((i >> s) & 1) == 0]
    return i, i + (1 << s)


def _boxplus_jitter(rng):
    """_f32_boxplus with every exp / log result moved one ulp up or down at random."""
    def j(v):
        up = rng.random(v.shape) < 0.5
        return np.where(up, np.nextafter(v, np.float32(np.inf)), np.nextafter(v, np.float32(-np.inf))).astype(np.float32)

    def f(a, b):
        a = np.clip(a, -LLR_MAX, LLR_MAX).astype(np.float32)
        b = np.clip(b, -LLR_MAX, LLR_MAX).astype(np.float32)
        out = j(np.log(np.float32(1) + j(np.exp(a + b)))).astype(np.float32)
        out -= j(np.log(j(np.exp(a)) + j(np.exp(b)))).astype(np.float32)
        return out.astype(np.float32)
    return f


def bp_decode_full(logits, frozen, num_iter, boxplus=False, ulp_jitter_seed=None):
    """Soft output -(Lm[0] + Rm[0]) of every position, fp32 [B, n] (logit convention; hard bit = soft > 0).
    frozen: uint8 [n], 1 = frozen.  ulp_jitter_seed (boxplus only): move every exp / log result by one ulp."""
    llr = -np.asarray(logits, dtype=np.float32)
    B, n = llr.shape
    m = int(np.log2(n))
    if boxplus:
        f = po._f32_boxplus if ulp_jitter_seed is None else _boxplus_jitter(np.random.default_rng(ulp_jitter_seed))
    else:
        f = po._f32
    L = [np.zeros((B, n), dtype=np.float32) for _ in range(m + 1)]
    R = [np.zeros((B, n), dtype=np.float32) for _ in range(m + 1)]
    L[m] = llr
    R[0][:] = np.where(np.asarray(frozen) != 0, LLR_MAX, np.float32(0))[None, :]
    pairs = [_pairs(n, s) for s in range(m)]
    for it in range(num_iter):
        for s in range(m - 1, -1, -1):
            i, j = pairs[s]
            a, b = L[s + 1][:, i], L[s + 1][:, j]
            ri, rj = R[s][:, i], R[s][:, j]
            L[s][:, i] = f(a, (b + rj).astype(np.float32))
            L[s][:, j] = (f(ri, a) + b).astype(np.float32)
        if it == num_iter - 1:
            break
        for s in range(m - 1):
            i, j = pairs[s]
            ri, rj = R[s][:, i], R[s][:, j]
            a, b = L[s + 1][:, i], L[s + 1][:, j]
            R[s + 1][:, i] = f(ri, (b + rj).astype(np.float32))
            R[s + 1][:, j] = (f(ri, a) + rj).astype(np.float32)
    return (-(L[0] + R[0])).astype(np.float32)


def _frozen_sets(n, rng):
    """(name, frozen positions): RM rule at rate 1/2, a random set, and the extremes k = 1, n-1, n."""
    sets = [("rm", po.rm_frozen_pos(n, n // 2)), ("random", np.sort(rng.choice(n, n // 2, replace=False))),
            ("k1", po.rm_frozen_pos(n, n - 1)), ("kn-1", po.rm_frozen_pos(n, 1)), ("kn", np.zeros(0, dtype=np.int64))]
    return [(name, np.asarray(fp, dtype=np.int64)) for name, fp in sets]


def _noiseless(rng, n, fp, B, mag=5.0):
    k = n - len(fp)
    u = rng.integers(0, 2, size=(B, k)).astype(np.uint8)
    c = po.encode(u, fp, n)
    return u, (mag * (2.0 * c - 1.0)).astype(np.float32)


# ---- CPU: the restatement's known answers, argument checks, constructors, CLI ------------------------------------------
def test_restatement_repetition_code():
    """n = 2, frozen = {0}: u1 is a repetition code; its soft output under min-sum is logit0 + logit1."""
    rng = np.random.default_rng(0)
    lg = rng.uniform(-30, 30, size=(1000, 2)).astype(np.float32)
    lg[:, 1] = rng.uniform(-200, 200, size=1000).astype(np.float32)
    for T in (1, 3, 20):
        soft = bp_decode_full(lg, np.array([1, 0], dtype=np.uint8), T)
        assert np.array_equal(soft[:, 1], lg[:, 0] + lg[:, 1]), T


@pytest.mark.parametrize("boxplus", [False, True])
def test_restatement_noiseless_recovery(boxplus):
    rng = np.random.default_rng(1)
    for n in NS:
        fp = po.rm_frozen_pos(n, n // 2)
        info = po.info_positions(fp, n)
        u, lg = _noiseless(rng, n, fp, 8)
        for T in (1, 20):
            soft = bp_decode_full(lg, po.frozen_vec(fp, n), T, boxplus=boxplus)
            assert np.array_equal((soft[:, info] > 0).astype(np.uint8), u), (n, T)


def test_restatement_ulp_jitter_moves_decisions_of_failing_words_mostly():
    """The calibration behind the boxplus bar: a 1-ulp jitter of exp / log rarely changes a word the restatement decodes
    correctly, and often changes one it fails."""
    rng = np.random.default_rng(2)
    n, k, B = 64, 32, 600
    fp = po.rm_frozen_pos(n, n - k)
    info, fz = po.info_positions(fp, n), po.frozen_vec(fp, n)
    from util import awgn_logits
    u, lg = awgn_logits(rng, n, k, fp, B, 1.0)
    ref = bp_decode_full(lg, fz, 20, boxplus=True)[:, info] > 0
    jit = bp_decode_full(lg, fz, 20, boxplus=True, ulp_jitter_seed=3)[:, info] > 0
    ok = (ref == (u != 0)).all(1)
    changed = (ref != jit).any(1)
    assert ok.sum() > 100 and (~ok).sum() > 20
    assert changed[ok].mean() < 0.01


def test_argument_checks_without_gpu():
    import d_kernels as dk
    lib = dk.lib()
    d = 256                                                             # never dereferenced: every call below fails early

    def call(n=64, B=5, T=20, mode=0, lg=d, fm=d, up=d, ui=None, sl=None, pos=None, k=32):
        return lib.polar_belief_decode_f32(lg, fm, n, B, T, mode, up, ui, sl, pos, k, None)
    before = lib.polar_launch_count()
    for kw in (dict(n=1), dict(n=0), dict(n=48), dict(n=2048), dict(T=0), dict(T=-1), dict(mode=2), dict(mode=-1),
               dict(B=-1), dict(lg=None), dict(fm=None), dict(up=None), dict(ui=d), dict(sl=d), dict(ui=d, pos=d, k=65),
               dict(sl=d, pos=d, k=-1)):
        assert call(**kw) == dk.POLAR_EINVAL, kw
    assert b"belief" in lib.polar_last_error()
    assert call(B=0, lg=None, fm=None, up=None) == dk.POLAR_OK
    assert call(B=0, n=1024, T=1, mode=1) == dk.POLAR_OK
    assert lib.polar_launch_count() == before


def test_constructor_checks():
    import torch
    from my_sn.fec.polar.dec import BP_Dec, Polar5GDecoder
    from my_sn.fec.polar.enc import Polar5GEncoder
    fp = po.rm_frozen_pos(64, 32)
    dec = BP_Dec(fp, 64)
    assert (dec.n, dec.k, dec.num_iter, dec.hard_out, dec.llr_max) == (64, 32, 20, True, 30.)
    assert np.array_equal(dec.info_pos, po.info_positions(fp, 64)) and dec.frozen_pos is fp
    d2 = BP_Dec(fp, 64, num_iter=5, hard_out=False, cn_type="minsum")
    assert d2.num_iter == 5 and d2.hard_out is False
    with pytest.raises(ValueError):
        BP_Dec(fp, 64, output_dtype=torch.int32)
    for kw in (dict(n=48), dict(n=2048, fp=po.rm_frozen_pos(2048, 1024)), dict(n=16), dict(num_iter=0),
               dict(num_iter=2.5), dict(hard_out=1), dict(cn_type="sum-product")):
        n = kw.pop("n", 64)
        with pytest.raises(AssertionError):
            BP_Dec(kw.pop("fp", fp), n, **kw)
    enc = Polar5GEncoder(100, 300)
    d5 = Polar5GDecoder(enc, "BP", num_iter=7)
    assert isinstance(d5._polar_dec, BP_Dec) and d5._polar_dec.num_iter == 7 and d5._polar_dec.n == enc.n_polar
    assert Polar5GDecoder(enc, "BP", 8, True)._return_crc_status
    with pytest.raises(ValueError):
        Polar5GDecoder(enc, "BPX")


def test_cli_accepts_bp():
    import importlib.util
    import os
    import sys
    from util import ROOT
    pkg = os.path.join(ROOT, "polar-code-pytorch-sionna_b200")
    saved = sys.modules.get("pyrallis")
    sys.modules["pyrallis"] = None                                      # the argparse fallback
    try:
        spec = importlib.util.spec_from_file_location("polar_main_cli_bp", os.path.join(pkg, "x_run_sn_polar", "main.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        c = m.parse_config(["--algos", "[sc,bp]", "--bp_iter", "5"])
    finally:
        if saved is None:
            sys.modules.pop("pyrallis", None)
        else:
            sys.modules["pyrallis"] = saved
    assert c.algos == ["sc", "bp"] and c.bp_iter == 5
    assert m.parse_config([]).bp_iter == 20


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _env():
    import torch
    import d_kernels as dk
    return torch, dk, torch.device("cuda", 0)


def _check_minsum(torch, dk, tables, lg, fp, T):
    """One min-sum decode of logits lg (numpy) against the restatement: soft, hard and packed outputs."""
    n = tables.n
    ref = bp_decode_full(lg, po.frozen_vec(fp, n), T)
    info = po.info_positions(fp, n)
    res = dk.belief_decode(torch.from_numpy(lg).to(tables.dev), tables, T, False, want_info=True, want_soft=True,
                           want_packed=True)
    soft = res["soft"].cpu().numpy()
    assert (soft == ref[:, info]).all()
    assert np.array_equal(res["u_info"].cpu().numpy(), (ref[:, info] > 0).astype(np.float32))
    bits = (ref > 0).astype(np.uint8)
    bits[:, po.frozen_vec(fp, n) != 0] = 0
    assert np.array_equal(unpack_words(res["u_packed"].cpu().numpy(), n), bits)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 2, 5, 20])
@pytest.mark.parametrize("n", NS)
def test_minsum_equals_restatement(n, T):
    torch, dk, dev = _env()
    from util import awgn_logits
    rng = np.random.default_rng(n * 100 + T)
    cpb = max(1, 512 // n)                                              # codewords per CTA
    for name, fp in _frozen_sets(n, rng):
        tables = dk.code_tables(fp, n, dev)
        k = n - len(fp)
        for ebno, B in ((0.0, 1), (1.5, 37), (4.0, 3 * cpb + 1)):
            _, lg = awgn_logits(rng, n, k, fp, B, ebno)
            _check_minsum(torch, dk, tables, lg, fp, T)


@pytest.mark.gpu
def test_minsum_large_batch_sample():
    """n = 1024, B = 2^18 (about 2.4 k waves of three CTAs per SM): a seeded sample of rows equals the restatement, and
    the same rows decoded in a small batch give the same outputs."""
    torch, dk, dev = _env()
    n, k, B, T = 1024, 512, 1 << 18, 5
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    _, _, lg = dk.awgn_frontend(tables, B, po.ebnodb2no(2.0, 2, k / n), seed=7)
    res = dk.belief_decode(lg, tables, T, False, want_info=True, want_soft=True, want_packed=True)
    rows = torch.from_numpy(np.sort(np.random.default_rng(8).choice(B, 4096, replace=False))).to(dev)
    ref = bp_decode_full(lg[rows].cpu().numpy(), po.frozen_vec(fp, n), T)
    info = po.info_positions(fp, n)
    assert (res["soft"][rows].cpu().numpy() == ref[:, info]).all()
    assert np.array_equal(res["u_info"][rows].cpu().numpy(), (ref[:, info] > 0).astype(np.float32))
    small = dk.belief_decode(lg[rows], tables, T, False, want_info=True, want_soft=True, want_packed=True)
    for key in ("soft", "u_info", "u_packed"):
        assert torch.equal(small[key], res[key][rows]), key


@pytest.mark.gpu
@pytest.mark.parametrize("n,B,ebno", [(64, 4000, 2.0), (256, 2000, 2.5), (1024, 800, 2.5)])
def test_boxplus_statistical(n, B, ebno):
    torch, dk, dev = _env()
    from util import awgn_logits
    rng = np.random.default_rng(n)
    k = n // 2
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    info = po.info_positions(fp, n)
    u, lg = awgn_logits(rng, n, k, fp, B, ebno)
    ref = bp_decode_full(lg, po.frozen_vec(fp, n), 20, boxplus=True)[:, info] > 0
    x = torch.from_numpy(lg).to(dev)
    got = dk.belief_decode(x, tables, 20, True)["u_info"].cpu().numpy() > 0
    ms = dk.belief_decode(x, tables, 20, False, want_info=False, want_soft=True)["soft"]
    bx = dk.belief_decode(x, tables, 20, True, want_info=False, want_soft=True)["soft"]
    ok = (ref == (u != 0)).all(1)
    assert ok.sum() > 0.3 * B
    assert (got[ok] == ref[ok]).all(1).mean() >= 0.99
    p_ref, p_got = 1 - ok.mean(), 1 - (got == (u != 0)).all(1).mean()
    p = 0.5 * (p_ref + p_got)
    assert abs(p_ref - p_got) <= 4 * np.sqrt(max(p * (1 - p), 1.0 / B) * 2 / B), (p_ref, p_got)
    assert not torch.equal(ms, bx)


@pytest.mark.gpu
@pytest.mark.parametrize("boxplus", [False, True])
def test_output_identities(boxplus):
    torch, dk, dev = _env()
    from util import awgn_logits
    n, k, B = 256, 128, 3001
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    _, lg = awgn_logits(np.random.default_rng(3), n, k, fp, B, 1.5)
    x = torch.from_numpy(lg).to(dev)
    res = dk.belief_decode(x, tables, 20, boxplus, want_info=True, want_soft=True, want_packed=True)
    assert torch.equal(res["u_info"], (res["soft"] > 0).float())
    bits = unpack_words(res["u_packed"].cpu().numpy(), n)
    assert np.array_equal(bits[:, po.info_positions(fp, n)], res["u_info"].cpu().numpy().astype(np.uint8))
    assert not bits[:, fp].any()
    # each output alone, into sentinel-filled buffers
    for want in ("u_info", "soft", "u_packed"):
        r = dk.belief_decode(x, tables, 20, boxplus, want_info=want == "u_info", want_soft=want == "soft",
                             want_packed=want == "u_packed")
        assert torch.equal(r[want], res[want]) and all(r[o] is None for o in res if o != want)
    buf = torch.full((B, n // 32), -1, dtype=torch.int32, device=dev)
    r = dk.belief_decode(x, tables, 20, boxplus, want_info=False, out_packed=buf)
    assert r["u_packed"] is buf and torch.equal(buf, res["u_packed"])
    si = torch.full((B, k), float("nan"), device=dev)
    sp = torch.full((B, k), float("nan"), device=dev)
    dk._call(dev, "polar_belief_decode_f32", dk.ptr(x), dk.ptr(tables.frozen_mask), n, B, 20, int(boxplus), None,
             dk.ptr(si), dk.ptr(sp), dk.ptr(tables.info_pos), k)
    assert torch.equal(si, res["u_info"]) and torch.equal(sp, res["soft"])
    # rows that are not 16-byte aligned are refused; the library keeps working
    flat = torch.empty(B * n + 1, device=dev)
    flat[1:].copy_(x.reshape(-1))
    lib = dk.lib()
    with torch.cuda.device(dev):
        rc = lib.polar_belief_decode_f32(ctypes.c_void_p(flat[1:].data_ptr()), dk.ptr(tables.frozen_mask), n, B, 20,
                                         int(boxplus), dk.ptr(buf), None, None, None, 0, dk.stream_ptr(dev))
    assert rc == dk.POLAR_EALIGN
    again = dk.belief_decode(flat[1:].view(B, n), tables, 20, boxplus, want_info=False, want_packed=True)   # realigned copy
    assert torch.equal(again["u_packed"], res["u_packed"])


@pytest.mark.gpu
def test_cuda_graph_capture_and_replay():
    torch, dk, dev = _env()
    n, k, B = 1024, 512, 4096
    fp = po.rm_frozen_pos(n, n - k)
    tables = dk.code_tables(fp, n, dev)
    no = po.ebnodb2no(2.0, 2, k / n)
    _, _, lg1 = dk.awgn_frontend(tables, B, no, seed=1)
    _, _, lg2 = dk.awgn_frontend(tables, B, no, seed=2)
    x = lg1.clone()
    soft = torch.empty((B, k), device=dev)
    run = lambda: dk._call(dev, "polar_belief_decode_f32", dk.ptr(x), dk.ptr(tables.frozen_mask), n, B, 20, 1, None, None,
                           dk.ptr(soft), dk.ptr(tables.info_pos), k)
    run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    x.copy_(lg2)
    g.replay()
    torch.cuda.synchronize()
    want = dk.belief_decode(lg2, tables, 20, True, want_info=False, want_soft=True)["soft"]
    assert torch.equal(soft, want)


@pytest.mark.gpu
def test_bp_dec_forward_shapes_and_hosts():
    torch, dk, dev = _env()
    from my_sn.fec.polar.dec import BP_Dec
    from util import awgn_logits
    n, k = 128, 64
    fp = po.rm_frozen_pos(n, n - k)
    _, lg = awgn_logits(np.random.default_rng(4), n, k, fp, 60, 2.0)
    x = torch.from_numpy(lg).reshape(3, 4, 5, n)
    hard, soft = BP_Dec(fp, n, num_iter=10), BP_Dec(fp, n, num_iter=10, hard_out=False, output_dtype=torch.float64)
    h_cpu, s_gpu = hard(x), soft(x.to(dev))
    assert h_cpu.shape == (3, 4, 5, k) and h_cpu.device.type == "cpu" and h_cpu.dtype == torch.float32
    assert s_gpu.shape == (3, 4, 5, k) and s_gpu.is_cuda and s_gpu.dtype == torch.float64
    from my_sn.sim import hard_decisions
    assert torch.equal(hard_decisions(s_gpu.float()).cpu(), h_cpu)
    tables = dk.code_tables(fp, n, dev)
    want = dk.belief_decode(x.to(dev), tables, 10, True, want_info=False, want_soft=True)["soft"]
    assert torch.equal(s_gpu.float().reshape(-1, k), want)
    packed = hard.decode_packed(x.to(dev), tables)
    assert np.array_equal(unpack_words(packed.cpu().numpy(), n)[:, po.info_positions(fp, n)],
                          h_cpu.reshape(-1, k).numpy().astype(np.uint8))


_STOP_CASES = (dict(max_mc_iter=7, target_block_errs=500), dict(max_mc_iter=5, target_bit_errs=2000),
               dict(max_mc_iter=3), dict(max_mc_iter=1, target_block_errs=1))


def _assert_loops_agree(torch, sim, mk, ebnos, bs, k):
    for kw in _STOP_CASES:
        host, devm = mk(99), mk(99)
        ber_h, bler_h = sim.sim_ber(host, ebnos, bs, verbose=False, on_device=False, **kw)
        ber_d, bler_d, cnt, status, iters = sim.sim_ber_device(devm, ebnos, bs, verbose=False, return_counters=True, **kw)
        assert torch.equal(ber_h, ber_d) and torch.equal(bler_h, bler_d), kw
        assert host._offset == devm._offset
        assert (cnt[:, 2] == cnt[:, 3] * k).all()


@pytest.mark.gpu
@pytest.mark.parametrize("cn_type", ["boxplus", "minsum"])
def test_device_loop_equals_host_loop(cn_type):
    torch, dk, dev = _env()
    from my_sn.fec.polar.dec import BP_Dec
    from polar.enc import PolarEncoder
    from z_sys_model.awgn_model import System_AWGN_model
    import my_sn.sim as sim
    n, k = 256, 128
    fp = po.rm_frozen_pos(n, n - k)
    mk = lambda seed, **kw: System_AWGN_model(n, k, PolarEncoder(fp, n, None), BP_Dec(fp, n, cn_type=cn_type, **kw), seed=seed)
    ebnos = np.array([0.0, 1.5, 3.0, 4.5, 9.0, 10.0], dtype=np.float32)
    _assert_loops_agree(torch, sim, mk, ebnos, 3000, k)
    # soft output + hard decisions in the host loop == hard output
    a = sim.sim_ber(mk(5), ebnos[:4], 3000, 3, verbose=False, on_device=False)
    b = sim.sim_ber(mk(5, hard_out=False), ebnos[:4], 3000, 3, soft_estimates=True, verbose=False)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ---- 5G ----------------------------------------------------------------------------------------------------------------
# none (64, 128), puncturing (100, 300), shortening (200, 400), repetition (300, 1088), from test_gpu_nr5g_link.CODES
NR_CODES = [(64, 128), (100, 300), (200, 400), (300, 1088), (40, 70)]


@pytest.mark.gpu
@pytest.mark.parametrize("k,e", NR_CODES)
def test_5g_bp(k, e):
    torch, dk, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.crc import CRCDecoder
    from my_sn.fec.polar.dec import Polar5GDecoder, BP_Dec
    from z_sys_model.awgn_model import System_AWGN_model
    enc = Polar5GEncoder(k, e)
    dec = Polar5GDecoder(enc, "BP", num_iter=20)
    model = System_AWGN_model(e, k, enc, dec, seed=5)
    bits, bits_hat = model(batch_size=2000, ebno_db=40.0)
    assert bits.shape == (2000, k) and torch.equal(bits, bits_hat)
    # the 5G decoder is rate recovery followed by BP_Dec, bit for bit, on noisy channel logits
    plan = enc.frontend_plan(dev)
    u_packed, _, lg = dk.nr5g_awgn_frontend(plan, 3000, po.ebnodb2no(0.5, 2, k / e), seed=9)
    u = dk.unpack_info(u_packed, plan.payload_pos_d, plan.n)
    ref_crc = BP_Dec(enc._frozen_pos, enc.n_polar, num_iter=20)(dec.rate_recover(lg))       # payload + CRC bits
    ref = ref_crc[:, :k]
    got = dec(lg)
    assert torch.equal(got, ref) and (got != u).any()                   # noisy enough that some words fail
    # CRC status: the CRC check of the BP decision (payload + CRC bits).  BP's hard decisions need not form a codeword,
    # so a correct payload can come with wrong CRC bits; the status is that of the decision, not of the payload.
    u_hat, status = Polar5GDecoder(enc, "BP", return_crc_status=True)(lg)
    _, ref_status = CRCDecoder(enc.enc_crc)(ref_crc)
    assert torch.equal(u_hat, ref) and status.shape == (3000,)
    assert torch.equal(status, ref_status.reshape(-1).to(status.dtype))
    _, _, lg_clean = dk.nr5g_awgn_frontend(plan, 500, po.ebnodb2no(40.0, 2, k / e), seed=10)
    _, st_clean = Polar5GDecoder(enc, "BP", return_crc_status=True)(lg_clean)
    assert bool((st_clean == 1).all())


@pytest.mark.gpu
@pytest.mark.parametrize("k,e", [(100, 300), (40, 70)])
def test_5g_device_loop_equals_host_loop(k, e):
    torch, dk, dev = _env()
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    from z_sys_model.awgn_model import System_AWGN_model
    import my_sn.sim as sim
    enc = Polar5GEncoder(k, e)
    mk = lambda seed: System_AWGN_model(e, k, enc, Polar5GDecoder(enc, "BP", num_iter=20), seed=seed)
    _assert_loops_agree(torch, sim, mk, np.array([-1.0, 1.0, 2.5, 4.0, 9.0, 10.0], dtype=np.float32), 3000, k)


@pytest.mark.gpu
def test_cli_bp_curve(tmp_path, monkeypatch):
    import importlib.util
    import os
    from util import ROOT
    pkg = os.path.join(ROOT, "polar-code-pytorch-sionna_b200")
    spec = importlib.util.spec_from_file_location("polar_main_cli_bp_gpu", os.path.join(pkg, "x_run_sn_polar", "main.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    c = m.parse_config(["--k", "32", "--n", "64", "--algos", "[bp]", "--bs", "100", "--mc_iter", "1"])
    monkeypatch.chdir(tmp_path)                                         # main() saves its plot under the working directory
    plot = m.main(c)
    names = [s for s in plot.legend if "BLER" in s]
    assert len(names) == 2 and names[0].startswith("SC") and names[1].startswith("BP-20"), plot.legend
