"""Generate tests/golden/*.npz by running the UNMODIFIED reference (build container only) and, in the
same pass, validate oracle/polar_oracle.py against it.  Run:  python oracle/gen_golden.py
Committed so the fixtures are reproducible; the fixtures (not this script) travel to the GPU box.
"""
import hashlib
import os
import random
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import ref_harness  # noqa: E402

ref_harness.install()
import torch as tc  # noqa: E402

from oracle import polar_oracle as po  # noqa: E402

from polar.froze import get_Kern_frozen_bits  # noqa: E402  (reference)
from polar.polar_sc import SC_Dec  # noqa: E402
from polar.polar_scl import SCL_Dec  # noqa: E402
from polar.enc import PolarEncoder as XEnc  # noqa: E402
from my_sn.fec.polar.enc import PolarEncoder as MyEnc  # noqa: E402
from my_sn.fec.polar.utils import generate_5g_ranking  # noqa: E402
from my_sn.fec.crc import CRCEncoder, CRCDecoder  # noqa: E402
from my_sn.trans import mapping, ebno as ref_ebno  # noqa: E402
from my_sn.trans.channel import awgn as ref_awgn  # noqa: E402
from my_sn.sim import sim_ber  # noqa: E402
from z_sys_model.awgn_model import System_AWGN_model  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)
F2 = tc.tensor([[1, 0], [1, 1]], dtype=tc.float32)


def set_seed(seed):  # main.py:25-29
    np.random.seed(seed)
    random.seed(seed)
    tc.manual_seed(seed)


def sha12(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:12]


def save(name, **kw):
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **kw)
    print("wrote %-28s %8.1f KB" % (name + ".npz", os.path.getsize(path) / 1024))


def ref_logits(n, k, frozen_pos, G, bs, ebno_db):
    """Reference front end, step by step (awgn_model.py:33-41) so the logits can be captured."""
    enc = XEnc(frozen_pos, n, G)
    model = System_AWGN_model(n, k, enc, None)
    no = ref_ebno.ebnodb2no(tc.tensor(float(ebno_db)), 2, k / n)
    bits = model.binary_src([bs, k])
    cw = enc(bits)
    x = model.mapper(cw)
    y = model.awgn_channel([x, no])
    llr = model.demapper([y, no])
    return bits.numpy(), cw.numpy(), llr.numpy().astype(np.float32)


# ------------------------------------------------------------------------------------------------
def gen_frozen():
    out = {}
    for n in (8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096):
        _, _, fp = get_Kern_frozen_bits(n, n // 2, F2)
        fp = fp.numpy().astype(np.int64)
        out["rm_%d_%d" % (n, n // 2)] = fp
        assert np.array_equal(po.rm_frozen_pos(n, n // 2), fp), n
        print("rm n=%d k=%d sha1=%s" % (n, n // 2, sha12(fp)))
    for (n, k) in ((64, 20), (128, 100), (1024, 256), (1024, 768)):
        _, _, fp = get_Kern_frozen_bits(n, n - k, F2)
        out["rm_%d_%d" % (n, k)] = fp.numpy().astype(np.int64)
        assert np.array_equal(po.rm_frozen_pos(n, n - k), out["rm_%d_%d" % (n, k)])
    for (k, n) in ((32, 64), (64, 128), (512, 1024), (100, 256), (501 + 11, 1024)):
        fp, ip = generate_5g_ranking(k, n)
        out["g5_%d_%d" % (n, k)] = np.asarray(fp, dtype=np.int64)
        print("5g n=%d k=%d sha1=%s" % (n, k, sha12(out["g5_%d_%d" % (n, k)])))
    out["cpu_capability"] = np.array(tc.backends.cpu.get_cpu_capability())
    out["torch_version"] = np.array(tc.__version__)
    save("frozen_sets", **out)
    return out


def gen_enc(fz):
    out = {}
    for (n, k, bs) in ((8, 4, 16), (64, 32, 64), (256, 128, 64), (1024, 512, 64), (4096, 2048, 8)):
        fp = fz["rm_%d_%d" % (n, k)]
        G, _, fpt = get_Kern_frozen_bits(n, n - k, F2)
        set_seed(100 + n)
        u = tc.randint(0, 2, (bs, k)).to(tc.float32)
        c1 = XEnc(fpt, n, G)(u).numpy()
        c2 = MyEnc(fp, n)(u).numpy()
        assert np.array_equal(c1, c2)
        assert np.array_equal(po.encode(u.numpy(), fp, n), c1.astype(np.uint8))
        out["u_%d" % n] = u.numpy().astype(np.uint8)
        out["c_%d" % n] = c1.astype(np.uint8)
    save("enc", **out)


EDGE16 = np.array([  # SURVEY A4 edge vectors (n=16, k=8)
    [+0.0] * 16, [-0.0] * 16, [100.0] * 16, [-100.0] * 16, [np.inf] * 16, [1e-30] * 16,
    [5, -7, 0, 0, 40, -40, 1, 1, -1, -1, 30, 30, -30, 30.0001, 2, -2],
], dtype=np.float32)


def gen_sc(fz):
    for (n, k, bs, ebno_db, key) in ((16, 8, 512, 2.0, "rm"), (64, 32, 512, 2.0, "rm"), (64, 32, 256, 2.0, "g5"),
                                     (128, 100, 256, 4.0, "rm"), (256, 128, 256, 3.0, "rm"),
                                     (1024, 512, 128, 4.0, "rm"), (1024, 512, 64, 2.5, "g5"),
                                     (1024, 256, 32, 1.0, "rm"), (1024, 768, 32, 5.0, "rm"),
                                     (2048, 1024, 32, 4.5, "rm"), (4096, 2048, 16, 5.0, "rm")):
        fp = fz["%s_%d_%d" % (key, n, k)]
        G = tc.from_numpy(po.arikan_G(n))
        set_seed(200 + n + k)
        bits, cw, llr = ref_logits(n, k, fp, G, bs, ebno_db)
        # add integer-quantised rows (ties / zeros) and, for n=16, the edge vectors
        q = np.round(llr[: bs // 4] * 0.5).astype(np.float32)
        rows = [llr, q]
        if n == 16:
            rows.append(EDGE16)
        logits = np.concatenate(rows, axis=0)
        dec = SC_Dec(fp, n)
        t0 = time.time()
        u_ref = dec(tc.from_numpy(logits)).numpy()
        dt = time.time() - t0
        u_or = po.sc_decode(logits, fp, n)
        assert np.array_equal(u_ref, u_or), ("SC oracle mismatch", n, k)
        bler = np.mean(np.any(u_ref[:bs] != bits, axis=1))
        print("sc %s n=%d k=%d rows=%d ref %.1fs  BLER(ref)=%.3f  oracle==ref" % (key, n, k, logits.shape[0], dt, bler))
        save("sc_%s_%d_%d" % (key, n, k), logits=logits, frozen_pos=fp, u_hat=u_ref.astype(np.uint8),
             bits=bits.astype(np.uint8), ebno_db=np.float32(ebno_db))


def gen_sc_boxplus(fz):
    """SURVEY 8f N2: the Sionna-style boxplus SC decoder (my_sn/fec/polar/dec.py:13-157).  Statistical fixture: the
    reference's decisions on AWGN words; the numpy restatement must agree on (almost) every codeword."""
    from my_sn.fec.polar.dec import SC_Dec as MySC
    # keep: codewords stored (the first ones of the batch), so that every fixture stays under 1 MB
    for (n, k, bs, ebno_db, keep) in ((64, 32, 2000, 2.0, 2000), (256, 128, 1000, 2.5, 1000), (1024, 512, 400, 3.0, 240)):
        fp = fz["rm_%d_%d" % (n, k)]
        G = tc.from_numpy(po.arikan_G(n))
        set_seed(900 + n)
        bits, cw, llr = ref_logits(n, k, fp, G, bs, ebno_db)
        dec = MySC(fp, n)
        u_ref = dec(tc.from_numpy(llr)).numpy()
        u_or = po.sc_decode_boxplus_full(llr, po.frozen_vec(fp, n))[:, po.info_positions(fp, n)]
        u_ms = po.sc_decode(llr, fp, n)
        agree = np.mean(np.all(u_ref == u_or, axis=1))
        print("sc-boxplus n=%d k=%d: BLER ref %.4f numpy-restatement %.4f min-sum %.4f | codewords identical to the restatement: %.4f"
              % (n, k, np.mean(np.any(u_ref != bits, axis=1)), np.mean(np.any(u_or != bits, axis=1)),
                 np.mean(np.any(u_ms != bits, axis=1)), agree))
        assert agree > 0.995
        save("scbp_rm_%d_%d" % (n, k), logits=llr[:keep], frozen_pos=fp, u_hat=u_ref[:keep].astype(np.uint8),
             bits=bits[:keep].astype(np.uint8), ebno_db=np.float32(ebno_db))


def gen_scl_boxplus(fz):
    """SURVEY 8f N2 (list decoder): the reference's my_sn SCL_Dec (exact boxplus, numpy float64) with use_fast_scl False
    (leaf-level path metrics = the arithmetic of polar_scl_decode_boxplus) and True (its default node shortcuts)."""
    from my_sn.fec.polar.dec import SCL_Dec as MySCL
    for (n, k, L, bs, ebno_db, crc) in ((64, 32, 8, 300, 2.0, None), (128, 64, 4, 200, 2.0, None), (256, 128, 8, 60, 2.5, "CRC11")):
        fp = fz["rm_%d_%d" % (n, k)]
        G = tc.from_numpy(po.arikan_G(n))
        set_seed(1200 + n)
        bits, cw, llr = ref_logits(n, k, fp, G, bs, ebno_db)
        res = {}
        for fast in (False, True):
            dec = MySCL(fp, n, list_size=L, crc_degree=crc, use_fast_scl=fast)
            res[fast] = dec(tc.from_numpy(llr)).numpy().astype(np.uint8)
        same = np.mean(np.all(res[False] == res[True], axis=1))
        print("scl-boxplus n=%d L=%d crc=%s: BLER slow %.4f fast %.4f, identical codewords %.4f" %
              (n, L, crc, np.mean(np.any(res[False] != bits, axis=1)), np.mean(np.any(res[True] != bits, axis=1)), same))
        save("sclbp_rm_%d_%d_L%d" % (n, k, L), logits=llr, frozen_pos=fp, u_hat=res[False], u_hat_fast=res[True],
             bits=bits.astype(np.uint8), crc_degree=np.array(crc if crc else ""), list_size=np.int64(L))


def gen_osd(fz):
    """SURVEY 8f N4: the reference's OSDecoder (my_sn/fec/osd/dec.py:8-192) on polar codes (its G = the encoder applied
    to the identity, dec.py:40-42).  The numpy restatement must return the reference's codewords."""
    from my_sn.fec.osd.dec import OSDecoder
    out = {}
    for (n, k, t, bs, no) in ((16, 8, 3, 120, 0.8), (32, 16, 2, 160, 0.6), (64, 32, 1, 160, 0.7), (64, 32, 2, 48, 0.7),
                              (128, 64, 1, 48, 0.8), (128, 100, 0, 64, 0.3)):
        fp = fz["rm_%d_%d" % (n, k)] if "rm_%d_%d" % (n, k) in fz else po.rm_frozen_pos(n, n - k)
        enc = MyEnc(fp, n)
        dec = OSDecoder(t=t, encoder=enc)
        set_seed(1700 + n + t)
        u = tc.randint(0, 2, (bs, k)).float()
        c = enc(u)
        y = (1 - 2 * c) + tc.randn(bs, n) * float(np.sqrt(no))
        logit = (-2 * y / no).float()
        # row 0: |llr| up to 95 -- exp() overflows to inf in fp32 above 88.7, so wrong decisions there cost inf (dec.py:78).
        # (Magnitudes at the +-100 clip would tie, and torch.argsort leaves the order of ties open.)
        logit[0] = logit[0] * (95.0 / float(logit[0].abs().max()))
        c_ref = dec(logit).numpy().astype(np.uint8)
        gm = dec._gm.numpy().astype(np.uint8)
        got, d, gap = po.osd_decode(logit.numpy(), gm, t)
        bad = (got != c_ref).any(axis=1)
        print("osd n=%d k=%d t=%d: BLER %.3f, restatement differs on %d of %d (smallest candidate gap %.2e)" %
              (n, k, t, float((c_ref != c.numpy()).any(axis=1).mean()), int(bad.sum()), bs, gap.min()))
        assert not bad.any()
        key = "%d_%d_t%d" % (n, k, t)
        out["logits_" + key] = logit.numpy(); out["gm_" + key] = gm; out["c_hat_" + key] = c_ref
        out["c_tx_" + key] = c.numpy().astype(np.uint8); out["gap_" + key] = gap
    save("osd", **out)


def gen_5g():
    """SURVEY 8f N3: 5G rate matching (my_sn/fec/polar/enc.py:115-392) and rate recovery (dec.py:539-667) of the reference:
    index plans, encoded codewords and de-rate-matched decoder inputs for puncturing, shortening and repetition."""
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    cfgs = [(12, 160), (20, 64), (32, 64), (40, 100), (64, 128), (64, 200), (100, 150), (100, 300), (200, 256), (256, 512),
            (300, 1088), (500, 600), (500, 1024), (700, 1000), (1013, 1088), (57, 70), (33, 45), (150, 400)]
    out = {"cfgs": np.array(cfgs, dtype=np.int64)}
    rng = np.random.default_rng(5)
    for (k, n) in cfgs:
        enc = Polar5GEncoder(k, n)
        key = "%d_%d" % (k, n)
        out["npolar_" + key] = np.int64(enc.n_polar)
        out["crclen_" + key] = np.int64(enc.enc_crc.crc_length)
        out["frozen_" + key] = np.asarray(enc._frozen_pos, dtype=np.int64)
        out["idx_" + key] = np.asarray(enc._ind_rate_matching, dtype=np.int64)
        u = rng.integers(0, 2, (6, k)).astype(np.float32)
        out["u_" + key] = u.astype(np.uint8)
        out["c_" + key] = enc(tc.from_numpy(u)).numpy().astype(np.uint8)
        dec = Polar5GDecoder(enc, dec_type="SC")
        grab = {}

        class Grab(tc.nn.Module):
            def forward(self, x):
                grab["x"] = x.clone()
                return tc.zeros([x.shape[0], enc.k_polar])
        dec._polar_dec = Grab()
        llr = (rng.standard_normal((4, n)) * 5).astype(np.float32)
        dec(tc.from_numpy(llr))
        out["llr_" + key] = llr
        out["dem_" + key] = grab["x"].numpy().astype(np.float32)
        print("5g k=%d n=%d: n_polar=%d crc=%d" % (k, n, enc.n_polar, enc.enc_crc.crc_length))
    # downlink plan (forward raises in the reference; the tables are still built)
    for (k, n) in [(30, 108), (140, 576)]:
        enc = Polar5GEncoder(k, n, channel_type="downlink")
        key = "dl_%d_%d" % (k, n)
        out["npolar_" + key] = np.int64(enc.n_polar)
        out["frozen_" + key] = np.asarray(enc._frozen_pos, dtype=np.int64)
        out["idx_" + key] = np.asarray(enc._ind_rate_matching, dtype=np.int64)
        out["iil_" + key] = np.asarray(enc._ind_input_int, dtype=np.int64)
    save("nr5g", **out)


def packbits(a):
    return np.packbits(a.astype(np.uint8), axis=-1, bitorder="little")


def gen_scl(fz):
    cases = ((64, 32, 2, 96, 2.0, "rm"), (64, 32, 4, 96, 2.0, "rm"), (64, 32, 8, 96, 2.0, "rm"),
             (64, 32, 16, 48, 2.0, "rm"), (64, 32, 32, 48, 2.0, "rm"), (64, 32, 1, 48, 2.0, "rm"),
             (128, 100, 8, 48, 4.5, "rm"),
             (256, 128, 4, 48, 2.5, "rm"), (256, 128, 8, 48, 2.5, "rm"),
             (1024, 512, 8, 48, 3.0, "rm"), (1024, 512, 4, 24, 3.0, "rm"), (1024, 512, 2, 16, 3.0, "rm"),
             (1024, 512, 8, 24, 2.0, "g5"),
             (2048, 1024, 32, 3, 3.5, "rm"), (4096, 2048, 4, 4, 4.0, "rm"))
    for (n, k, L, bs, ebno_db, key) in cases:
        fp = fz["%s_%d_%d" % (key, n, k)]
        G = tc.from_numpy(po.arikan_G(n))
        set_seed(300 + n + k)          # same logits for every L of a given (n, k)
        bits, cw, llr = ref_logits(n, k, fp, G, bs, ebno_db)
        dec = SCL_Dec(fp, n, list_size=L)
        t0 = time.time()
        u_best_ref = dec(tc.from_numpy(llr)).numpy()
        dt = time.time() - t0
        # full list state left on the decoder object by forward (polar_scl.py:203-206)
        u_list_ref = dec.msg_uhat[:, :, 0, :].astype(np.uint8)      # [B, 2L, n], pm-ascending
        pm_ref = dec.msg_pm.copy()                                   # [B, 2L]
        u_a, pm_a = po.scl_decode_full(llr, po.frozen_vec(fp, n), L)
        u_b, pm_b = po.scl_decode_full(llr, po.frozen_vec(fp, n), L, use_log1p=True)
        u_c, pm_c = po.scl_decode_full(llr, po.frozen_vec(fp, n), L, stable_sort=False)
        info = po.info_positions(fp, n)
        best_ok = np.array_equal(u_a[:, 0, info].astype(np.float32), u_best_ref)
        # reference's 2L sorted PMs are the L PMs duplicated pairwise (SURVEY A9)
        pm_ref_sorted = np.sort(pm_ref, axis=1)
        pm_pairs = pm_ref_sorted[:, 0::2]
        best_pm_rel = np.max(np.abs(pm_a[:, 0] - pm_pairs[:, 0]) / np.maximum(np.abs(pm_pairs[:, 0]), 1e-300))

        def setkey(u):  # order-independent fingerprint of a list
            return [frozenset(map(bytes, packbits(u[b]))) for b in range(u.shape[0])]
        s_ref, s_a, s_b, s_c = setkey(u_list_ref), setkey(u_a), setkey(u_b), setkey(u_c)
        robust = np.array([s_ref[b] == s_a[b] == s_b[b] == s_c[b] for b in range(bs)])
        pm_exact = np.array([np.array_equal(pm_a[b], pm_pairs[b]) for b in range(bs)])
        print("scl %s n=%d k=%d L=%d bs=%d ref %.1fs best_ok=%s bestPMrel=%.1e robust_lists=%d/%d pm_bitexact=%d/%d BLER=%.3f"
              % (key, n, k, L, bs, dt, best_ok, best_pm_rel, robust.sum(), bs, pm_exact.sum(), bs,
                 np.mean(np.any(u_best_ref != bits, axis=1))))
        assert best_ok, "SCL oracle best path mismatch"
        assert best_pm_rel < 1e-12
        save("scl_%s_%d_%d_L%d" % (key, n, k, L), logits=llr, frozen_pos=fp,
             u_best=u_best_ref.astype(np.uint8), pm=pm_pairs, u_list=packbits(u_list_ref[:, 0::1]),
             robust=robust, bits=bits.astype(np.uint8), ebno_db=np.float32(ebno_db))


def gen_crc(fz):
    out = {}
    # KAT (SURVEY A13)
    kat_in = np.array([1, 1, 0, 0, 1, 1, 1, 1, 1, 0, 0, 1, 0, 1, 1, 0, 0, 1, 0, 0, 0], dtype=np.float32)
    enc = CRCEncoder("CRC11", kat_in.shape[0])
    kat_out = enc(tc.from_numpy(kat_in)[None, :]).numpy()[0]
    print("CRC11 KAT parity:", kat_out[-11:].astype(int).tolist())
    assert np.array_equal(po.crc_encode(kat_in[None], "CRC11")[0], kat_out.astype(np.uint8))
    out["kat_in"] = kat_in.astype(np.uint8)
    out["kat_out"] = kat_out.astype(np.uint8)
    for deg in po.CRC_COEFFS:
        set_seed(7)
        k = 57
        b = tc.randint(0, 2, (32, k)).to(tc.float32)
        e = CRCEncoder(deg, k)
        y = e(b).numpy().astype(np.uint8)
        assert np.array_equal(po.crc_encode(b.numpy(), deg), y), deg
        ln = po.CRC_COEFFS[deg][0]
        d = CRCDecoder(CRCEncoder(deg, k + ln))
        ybad = y.copy()
        ybad[::2, 5] ^= 1
        _, ok = d(ybad.astype(np.float32))
        assert np.array_equal(ok[:, 0], po.crc_valid(ybad, deg)), deg
        out["in_" + deg] = b.numpy().astype(np.uint8)
        out["out_" + deg] = y
        out["bad_" + deg] = ybad
        out["ok_" + deg] = ok[:, 0]
    save("crc", **out)

    # CRC-aided SCL (composed oracle, SURVEY 8c): x_run SCL list -> my_sn dec.py:507-527 selection
    from my_sn.fec.polar.dec import SCL_Dec as MySCL
    for (n, k, L, deg, bs, ebno_db, key) in ((64, 32, 8, "CRC6", 96, 1.5, "rm"), (256, 128, 8, "CRC11", 64, 3.0, "rm"),
                                             (1024, 512, 8, "CRC11", 48, 3.75, "rm"), (1024, 512, 8, "CRC24C", 24, 3.75, "rm")):
        fp = fz["%s_%d_%d" % (key, n, k)]
        ln = po.CRC_COEFFS[deg][0]
        G = tc.from_numpy(po.arikan_G(n))
        set_seed(400 + n + ln)
        payload = tc.randint(0, 2, (bs, k - ln)).to(tc.float32)
        bits = CRCEncoder(deg, k - ln)(payload)                      # [bs, k] payload+parity
        enc = XEnc(fp, n, G)
        model = System_AWGN_model(n, k, enc, None)
        no = ref_ebno.ebnodb2no(tc.tensor(float(ebno_db)), 2, k / n)
        cw = enc(bits)
        llr = model.demapper([model.awgn_channel([model.mapper(cw), no]), no]).numpy().astype(np.float32)
        dec = SCL_Dec(fp, n, list_size=L)
        msg_uhat, msg_pm = dec._decode_np_batch(-1.0 * tc.from_numpy(llr))     # polar_scl.py:219-220
        my = MySCL(fp, n, list_size=L, crc_degree=deg)
        info = dec._info_pos
        u_list = msg_uhat[:, :, 0, :][:, :, info]
        _, valid = my._crc_decoder(u_list.astype(np.float32))                   # dec.py:516
        pm_pen = msg_pm + np.squeeze((1.0 - valid) * my._llr_max * my.k, axis=2)  # dec.py:517-518
        cand = np.argmin(pm_pen, axis=-1)                                       # dec.py:520
        u_sel = msg_uhat[np.arange(bs), cand, 0, :][:, info].astype(np.uint8)
        # oracle
        u_a, pm_a = po.scl_decode_full(llr, po.frozen_vec(fp, n), L)
        u_or, idx = po.scl_crc_select(u_a, pm_a, fp, n, deg)
        u_b, pm_b = po.scl_decode_full(llr, po.frozen_vec(fp, n), L, use_log1p=True)
        u_or_b, _ = po.scl_crc_select(u_b, pm_b, fp, n, deg)
        u_c, pm_c = po.scl_decode_full(llr, po.frozen_vec(fp, n), L, stable_sort=False)
        u_or_c, _ = po.scl_crc_select(u_c, pm_c, fp, n, deg)
        agree = np.all(u_or == u_sel, axis=1)
        robust = agree & np.all(u_or_b == u_sel, axis=1) & np.all(u_or_c == u_sel, axis=1)
        noaid = np.all(u_a[:, 0][:, info] == bits.numpy(), axis=1)
        print("scl+%s n=%d L=%d: oracle==composed-ref %d/%d, robust %d/%d, BLER aided %.3f vs unaided %.3f, crc-changed-choice %d"
              % (deg, n, L, agree.sum(), bs, robust.sum(), bs, np.mean(np.any(u_sel != bits.numpy(), axis=1)),
                 1 - noaid.mean(), int(np.sum(idx != 0))))
        save("sclcrc_%s_%d_%d_L%d_%s" % (key, n, k, L, deg), logits=llr, frozen_pos=fp, u_sel=u_sel,
             robust=robust, bits=bits.numpy().astype(np.uint8), crc_degree=np.array(deg), ebno_db=np.float32(ebno_db))


def gen_frontend():
    n, k, bs = 64, 32, 64
    set_seed(5)
    const = mapping.QamConstell(2)
    mapper = mapping.Mapper(constell=const)
    demap = mapping.Demapper(constell=const)
    cw = tc.randint(0, 2, (bs, n)).to(tc.float32)
    out = {"cw": cw.numpy().astype(np.uint8)}
    for ebno_db in (0.0, 3.0, 6.0):
        no = ref_ebno.ebnodb2no(tc.tensor(ebno_db), 2, k / n)
        x = mapper(cw)
        nr = tc.normal(mean=0, std=tc.sqrt(tc.tensor(0.5)), size=x.shape)
        ni = tc.normal(mean=0, std=tc.sqrt(tc.tensor(0.5)), size=x.shape)
        y = x + tc.complex(nr, ni) * tc.sqrt(no.to(tc.float32))
        llr = demap([y, no]).numpy()
        mine = po.qpsk_awgn_logits(cw.numpy(), nr.numpy(), ni.numpy(), float(no))
        err = np.max(np.abs(mine - llr))
        assert err < 2e-5 * max(1.0, np.max(np.abs(llr))), err
        assert np.array_equal(np.sign(mine), np.sign(llr))
        assert abs(po.ebnodb2no(ebno_db, 2, k / n) - float(no)) < 1e-7
        tag = "%d" % int(ebno_db)
        out["no_" + tag] = np.float32(no)
        out["nr_" + tag] = nr.numpy()
        out["ni_" + tag] = ni.numpy()
        out["llr_" + tag] = llr.astype(np.float32)
        print("frontend %.1f dB: closed form vs layer stack max abs diff %.2e (max |llr| %.1f)" % (ebno_db, err, np.max(np.abs(llr))))
    save("frontend", **out)


def gen_readme_kat(fz):
    """README command (readme.md:7) with main.py's seeding (main.py:55-59): the reference's only
    published result (the BLER plot).  Stores the curves; the oracle re-derives them in tests by
    drawing from the same torch-CPU mt19937 stream in the same call order (SURVEY 3.2)."""
    n, k, bs = 64, 32, 100
    ebno_dbs = np.arange(0, 5, 0.5)
    G, _, fp = get_Kern_frozen_bits(n, n - k, F2)
    res = {}
    for name, dec in (("sc", SC_Dec(fp, n)), ("scl8", SCL_Dec(fp, n, 8))):
        model = System_AWGN_model(n, k, XEnc(fp, n, G), dec)
        set_seed(42)
        ber, bler = sim_ber(model, ebno_dbs, bs, 1, target_block_errs=1000, verbose=False)
        res[name + "_ber"] = ber.numpy()
        res[name + "_bler"] = bler.numpy()
        print(name, "BLER", np.round(bler.numpy(), 3).tolist())
    save("readme_kat", ebno_dbs=ebno_dbs, frozen_pos=fp.numpy(), **res)


if __name__ == "__main__":
    which = sys.argv[1:] or ["frozen", "enc", "sc", "scbp", "nr5g", "sclbp", "scl", "crc", "frontend", "readme", "osd"]
    fz = gen_frozen() if "frozen" in which else dict(np.load(os.path.join(OUT, "frozen_sets.npz")))
    if "enc" in which:
        gen_enc(fz)
    if "frontend" in which:
        gen_frontend()
    if "readme" in which:
        gen_readme_kat(fz)
    if "crc" in which:
        gen_crc(fz)
    if "sc" in which:
        gen_sc(fz)
    if "scbp" in which:
        gen_sc_boxplus(fz)
    if "nr5g" in which:
        gen_5g()
    if "sclbp" in which:
        gen_scl_boxplus(fz)
    if "scl" in which:
        gen_scl(fz)
    if "osd" in which:
        gen_osd(fz)
