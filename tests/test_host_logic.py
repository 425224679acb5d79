"""CPU tests of the host-side logic: frozen-set construction, 5G ranking, CRC tables, packing helpers,
the reference call surface's argument checks, and that the C-ABI library loads and exports every symbol
include/polar_b200.h declares (no compute calls: there is no GPU here)."""
import ctypes
import hashlib
import os
import re
import subprocess

import numpy as np
import pytest

from util import golden, ROOT

PKG = os.path.join(ROOT, "polar-code-pytorch-sionna_b200")
LIB = os.path.join(PKG, "libpolar_b200.so")
SHA = {8: "69a9dc94b314", 16: "8acaf4773769", 32: "563716f9ce74", 64: "737f49d39c2f", 128: "65bde1d5fb3f",
       256: "b3950a1dfa94", 512: "1accab96ad9f", 1024: "6328351f152c", 2048: "8214d125add5", 4096: "a9616caf4c90"}  # SURVEY A1


def _sha(a):
    return hashlib.sha1(np.ascontiguousarray(a, dtype=np.int64).tobytes()).hexdigest()[:12]


def test_golden_frozen_sets_have_reference_fingerprints():
    fz = golden("frozen_sets")
    for n, h in SHA.items():
        assert _sha(fz["rm_%d_%d" % (n, n // 2)]) == h
    assert fz["rm_64_32"].tolist() == list(range(13)) + [16, 17, 18, 19, 20, 24] + list(range(32, 39)) + [40, 41, 42, 44, 48, 52]
    assert _sha(fz["g5_64_32"]) == "959cc8ff8790" and _sha(fz["g5_128_64"]) == "4cb9b4aee8b0" and _sha(fz["g5_1024_512"]) == "6d6017af8e33"


def test_get_kern_frozen_bits_matches_reference():
    import torch
    from polar.froze import get_Kern_frozen_bits, get_Kern_frozen_bits2
    from d_kernels import F2, F4, gen_arikan
    fz = golden("frozen_sets")
    same_host = str(fz["cpu_capability"]) == torch.backends.cpu.get_cpu_capability()
    for n in (8, 16, 64, 128, 1024):
        G, w, fp = get_Kern_frozen_bits(n, n // 2, F2)
        assert isinstance(fp, torch.Tensor) and fp.dtype == torch.int64 and G.shape == (n, n)
        i = np.arange(n)
        assert np.array_equal(G.cpu().numpy(), ((i[:, None] & i[None, :]) == i[None, :]).astype(np.float32))   # G[i,j]=1 <=> j subset i
        assert np.array_equal(w.cpu().numpy(), 2.0 ** np.array([bin(v).count("1") for v in i]))
        f = fp.numpy()
        # RM rule: every frozen row is at most as heavy as every info row (tie members are argsort's choice)
        wt = w.cpu().numpy()
        info = np.setdiff1d(i, f)
        assert wt[f].max() <= wt[info].min() and len(f) == n // 2
        if same_host:   # torch.argsort tie order depends on the CPU SIMD level (SURVEY A1 hazard)
            assert np.array_equal(f, fz["rm_%d_%d" % (n, n // 2)])
    assert torch.equal(gen_arikan(F2, 2), F4)
    G2, w2, fp2 = get_Kern_frozen_bits2(16, 8, F2.cpu().numpy())
    assert len(fp2) == 8 and np.array_equal(G2, get_Kern_frozen_bits(16, 8, F2)[0].cpu().numpy())
    with pytest.raises(AssertionError):
        get_Kern_frozen_bits(24, 12, F2)


def test_5g_ranking_and_rm_code():
    from my_sn.fec.polar.utils import generate_5g_ranking, generate_rm_code
    fz = golden("frozen_sets")
    for (k, n) in ((32, 64), (64, 128), (512, 1024), (100, 256)):
        fp, ip = generate_5g_ranking(k, n)
        assert np.array_equal(fp, fz["g5_%d_%d" % (n, k)])
        assert np.array_equal(np.sort(np.concatenate([fp, ip])), np.arange(n))
    assert generate_5g_ranking(32, 64)[0].tolist() == list(range(15)) + list(range(16, 22)) + [24, 25, 26] + list(range(32, 38)) + [40, 48]
    with pytest.raises(AssertionError):
        generate_5g_ranking(1024, 2048)
    fr, info, n, k, d = generate_rm_code(3, 6)
    assert (n, k, d) == (64, 42, 8)
    assert fr.tolist() == [0, 1, 2, 3, 4, 5, 6, 8, 9, 10, 12, 16, 17, 18, 20, 24, 32, 33, 34, 36, 40, 48]


def test_crc_encoder_decoder_match_reference():
    import torch
    from my_sn.fec.crc import CRCEncoder, CRCDecoder
    d = golden("crc")
    enc = CRCEncoder("CRC11", 21)
    out = enc(torch.from_numpy(d["kat_in"].astype(np.float32))[None])[0].numpy()
    assert out[-11:].astype(int).tolist() == [0, 0, 0, 1, 1, 1, 1, 0, 1, 1, 1]
    for deg, ln in (("CRC24A", 24), ("CRC24B", 24), ("CRC24C", 24), ("CRC16", 16), ("CRC11", 11), ("CRC6", 6)):
        e = CRCEncoder(deg, 57)
        assert e.crc_length == ln and e.k == 57 and e.n == 57 + ln
        y = e(torch.from_numpy(d["in_" + deg].astype(np.float32))).numpy().astype(np.uint8)
        assert np.array_equal(y, d["out_" + deg])
        dec = CRCDecoder(CRCEncoder(deg, 57 + ln))
        x, ok = dec(torch.from_numpy(d["bad_" + deg].astype(np.float32)))
        assert np.array_equal(ok[:, 0].numpy(), d["ok_" + deg]) and x.shape[-1] == 57
        # syndrome rows used by the fused CRC epilogue: XOR of rows at set bits == 0  <=>  valid
        chk = CRCEncoder(deg, 57 + ln)
        rows = chk.syndrome_rows(np.arange(57 + ln) * 2, 2 * (57 + ln))[::2]
        syn = np.bitwise_xor.reduce(np.where(d["bad_" + deg] != 0, rows[None, :], 0), axis=1)
        assert np.array_equal(syn == 0, d["ok_" + deg])
    with pytest.raises(ValueError):
        CRCEncoder("CRC7", 10)


def test_packing_helpers_and_code_tables_layout():
    import d_kernels as dk
    fp = np.array([0, 1, 2, 4, 33, 63])
    w = dk.frozen_mask_words(fp, 64)
    assert w.dtype == np.uint32 and w.tolist() == [0b10111, (1 << 1) | (1 << 31)]
    assert dk.frozen_mask_words(np.array([0, 3]), 8).tolist() == [0b1001]
    assert dk.words(8) == 1 and dk.words(32) == 1 and dk.words(1024) == 32
    import torch
    assert np.array_equal(dk.to_numpy_pos(torch.tensor([3, 1])), np.array([3, 1]))


def test_constructor_argument_checks_mirror_reference():
    import torch
    from polar.polar_scl import SCL_Dec
    from polar.polar_sc import SC_Dec
    from polar.enc import PolarEncoder
    from my_sn.fec.polar.dec import SCL_Dec as MySCL
    fp = golden("frozen_sets")["rm_16_8"]
    with pytest.raises(AssertionError, match="list_size must be a power of 2"):
        SCL_Dec(fp, 16, list_size=3)
    with pytest.raises(AssertionError, match="n must be a power of 2"):
        SCL_Dec(fp, 24)
    with pytest.raises(ValueError):
        SCL_Dec(fp, 16, output_dtype=torch.int8)
    with pytest.raises(ValueError):
        MySCL(fp, 16, return_crc_status=True)
    with pytest.raises(AssertionError):
        MySCL(fp, 16, crc_degree="CRC11")            # k=8 < 11 CRC bits
    with pytest.raises(Exception):
        SC_Dec(fp, 16, mode="bogus")
    d = SC_Dec(torch.from_numpy(fp), 16)
    assert d.k == 8 and d.n == 16 and d.llr_max == 30. and d.info_pos.tolist() == [7, 9, 10, 11, 12, 13, 14, 15]
    s = SCL_Dec(fp, 16, 32)
    assert (s.n, s.k, s.list_size) == (16, 8, 32)
    e = PolarEncoder(fp, 16, None)
    assert e.k == 8
    if not torch.cuda.is_available():                 # no CPU fallback: the product path must fail loudly
        with pytest.raises(RuntimeError, match="no CUDA device"):
            d(torch.zeros(2, 16))
        with pytest.raises(RuntimeError, match="no CUDA device"):
            e(torch.zeros(2, 8))


def test_library_exports_every_declared_symbol():
    assert os.path.exists(LIB), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    hdr = open(os.path.join(ROOT, "include", "polar_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(polar_[a-z0-9_]+)\s*\(", hdr))
    assert {"polar_sc_decode_f32", "polar_scl_decode", "polar_encode_packed", "polar_awgn_frontend",
            "polar_count_errors_packed", "polar_scl_workspace_bytes", "polar_last_error"} <= declared
    L = ctypes.CDLL(LIB)
    for name in sorted(declared):
        assert hasattr(L, name), name
    import d_kernels as dk
    assert set(dk._SIGNATURES) == declared            # the ctypes table covers exactly the header
    lib = dk.lib()
    assert b"sm_100a" in lib.polar_version()
    # argument validation happens before any CUDA call, so it is testable without a GPU
    assert lib.polar_sc_decode_f32(None, None, 24, 1, None, None, None, 0, None) == dk.POLAR_EINVAL
    assert b"power of two" in lib.polar_last_error()
    assert lib.polar_scl_decode(None, None, 64, 3, 1, None, None, None, 0, None, None, None, 0, None, 0, None) == dk.POLAR_EINVAL
    assert lib.polar_scl_decode(None, None, 8192, 8, 1, None, None, None, 0, None, None, None, 0, None, 0, None) == dk.POLAR_EINVAL
    assert lib.polar_encode_packed(None, 64, 1, None, None) == dk.POLAR_EINVAL
    assert lib.polar_sc_decode_f32(None, None, 64, 0, None, None, None, 0, None) == dk.POLAR_OK       # empty batch
    with pytest.raises(AssertionError):
        dk.check(dk.POLAR_EINVAL)


def test_library_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "-lelf", LIB], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


def test_register_subtree_decoder_on_host(tmp_path):
    """polar_common.cuh's SubTree<T> (the per-thread 32-leaf SC decoder) compiled as plain C++ vs the C oracle."""
    from oracle import c_oracle as co
    co.build()
    exe = str(tmp_path / "polar_subtree_check")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-I" + os.path.join(PKG, "csrc"),
                           os.path.join(ROOT, "tests", "host", "subtree_check.cpp"), "-o", exe,
                           "-L" + os.path.join(ROOT, "oracle"), "-lpolar_oracle",
                           "-Wl,-rpath," + os.path.join(ROOT, "oracle"), "-lpthread"])
    assert subprocess.run([exe], capture_output=True, text=True).stdout.strip().endswith("bad=0")


def test_5g_rate_matching_plans_match_reference():
    """SURVEY 8f N3 (host side): mother-code length, CRC choice, frozen set and the combined rate-matching gather index of
    Polar5GEncoder for puncturing / shortening / repetition configs, and the interleavers, against the reference's tables."""
    import numpy as np
    from util import golden
    from my_sn.fec.polar.enc import Polar5GEncoder
    from my_sn.fec.polar.dec import Polar5GDecoder
    g = golden("nr5g")
    for k, n in g["cfgs"]:
        key = "%d_%d" % (k, n)
        enc = Polar5GEncoder(int(k), int(n))
        assert enc.n_polar == int(g["npolar_" + key]) and enc.enc_crc.crc_length == int(g["crclen_" + key]), key
        assert np.array_equal(np.asarray(enc._frozen_pos), g["frozen_" + key]), key
        assert np.array_equal(enc._ind_rate_matching, g["idx_" + key]), key
        assert enc.k == k and enc.n == n and enc.k_polar == k + enc.enc_crc.crc_length
        # the fused rate-recovery plan reproduces the reference's de-rate-matched decoder input on the host
        dec = Polar5GDecoder(enc, dec_type="SC")               # construction is host-only
        s0, s1, fill = dec._plan
        llr = g["llr_" + key]
        out = np.where(s0 >= 0, llr[:, np.maximum(s0, 0)], fill[None, :]).astype(np.float32)
        out = out + np.where(s1 >= 0, llr[:, np.maximum(s1, 0)], np.float32(0)).astype(np.float32)
        assert np.array_equal(out, g["dem_" + key]), key
    for key in ("dl_30_108", "dl_140_576"):
        k, n = (int(v) for v in key.split("_")[1:])
        enc = Polar5GEncoder(k, n, channel_type="downlink")
        assert enc.n_polar == int(g["npolar_" + key])
        assert np.array_equal(np.asarray(enc._frozen_pos), g["frozen_" + key])
        assert np.array_equal(enc._ind_rate_matching, g["idx_" + key])
        assert np.array_equal(enc._ind_input_int, g["iil_" + key])
    import pytest
    with pytest.raises(ValueError):
        Polar5GEncoder(8, 64)
    with pytest.raises(AssertionError):
        Polar5GEncoder(100, 50)
    with pytest.raises(AssertionError):
        Polar5GEncoder(200, 400, channel_type="downlink")


def test_main_cli_fallback_parser_follows_the_annotations():
    """x_run_sn_polar/main.py without pyrallis: option types come from the dataclass annotations of config.py:5-26
    (`snr_end: float = 5` must accept 4.5, `algos` the reference's bracket list, `verbose` a boolean word)."""
    import importlib.util
    import sys
    for p in (PKG, os.path.join(PKG, "x_run_sn_polar")):
        if p not in sys.path:
            sys.path.insert(0, p)
    saved = sys.modules.get("pyrallis")
    sys.modules["pyrallis"] = None                      # force the argparse fallback
    try:
        spec = importlib.util.spec_from_file_location("polar_main_cli", os.path.join(PKG, "x_run_sn_polar", "main.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        c = m.parse_config(["--k", "1024", "--n", "2048", "--algos", "[sc,scl]", "--list_size", "32", "--snr_end", "4.5",
                            "--bs", "65536", "--mc_iter", "16", "--verbose", "true"])
    finally:
        if saved is None:
            sys.modules.pop("pyrallis", None)
        else:
            sys.modules["pyrallis"] = saved
    assert (c.k, c.n, c.list_size, c.bs, c.mc_iter) == (1024, 2048, 32, 65536, 16)
    assert c.snr_end == 4.5 and isinstance(c.snr_end, float)
    assert c.algos == ["sc", "scl"] and c.verbose is True
    d = m.parse_config([])
    assert (d.k, d.n, d.bs, d.snr_end, d.seed) == (32, 64, 3, 5, 42)


def test_sweep_planner_of_the_device_monte_carlo_loop():
    """my_sn/sim.py::SweepPlanner: which (point, iteration) items the device loop packs into one decoder launch.  A plan
    crosses into the next SNR point only where the current one is certain (3 sigma) to stop; a wrong plan can never change
    a result (the control kernel ignores items the sequential loop would not have run), it only wastes the ignored items."""
    from my_sn.sim import SweepPlanner
    start = (0, 0, (0.0, 0.0), (0.0, 0.0))
    # configs[3]: 65536 codewords per iteration, target 1000 block errors, every point far above it
    p = SweepPlanner(9, None, 1000, 16, per_iter_max=(0.5 * 65536 * 1024, 65536.0))
    items, after = p.plan(start, 32)
    assert items == [0, 1, 2, 3] and after is None          # chained lower bound 65536 x 0.3^j: certain for 3 points, the 4th is open
    p.finished_point(1, 3 * 10 ** 7, 65530)
    items, after = p.plan((4, 0, (0.0, 0.0), (0.0, 0.0)), 32)
    assert items == [4, 5, 6, 7] and after is None
    p.finished_point(1, 10 ** 7, 45000)
    items, after = p.plan((8, 0, (0.0, 0.0), (0.0, 0.0)), 32)
    assert items == [8] and after == "done"
    # waterfall region: 150 block errors per iteration known at this point -> 6 or 7 more iterations, uncertain which
    p = SweepPlanner(9, None, 1000, 16, per_iter_max=(1e9, 65536.0))
    items, after = p.plan((3, 1, (900.0, 150.0), (900.0, 150.0)), 32)
    assert set(items) == {3} and 4 <= len(items) <= 6 and after is None     # up to the earliest possible stop, then wait
    # no targets: the whole sweep is certain -- groups are cut by size only and chain across points
    p = SweepPlanner(3, None, None, 16, per_iter_max=(1.0, 1.0))
    items, after = p.plan(start, 8)
    assert items == [0] * 8 and after[:2] == (0, 8)
    items, after = p.plan(after, 12)
    assert items == [0] * 8 + [1] * 4 and after[:2] == (1, 4)
    items, after = p.plan((2, 10, (0.0, 0.0), (0.0, 0.0)), 32)
    assert items == [2] * 6 and after == "done"
    # a bit-error target decides as well; max_mc_iter caps every point
    p = SweepPlanner(2, 5000, None, 4, per_iter_max=(1e6, 1e3))
    items, after = p.plan((0, 1, (4000.0, 1.0), (4000.0, 1.0)), 32)
    assert items[:1] == [0] and items.count(0) == 1          # 8000 predicted bit errors against 5000: stops after one more
    p = SweepPlanner(2, None, 10 ** 6, 12, per_iter_max=(512 * 64 * 0.5, 512.0))
    items, after = p.plan(start, 32)
    assert items == [0] * 12 + [1] * 12 and after == "done"  # target out of reach: max_mc_iter iterations per point


def test_encoder_rejects_non_arikan_generator():
    """ADVICE r01: PolarEncoder applies the Arikan butterfly; any other G must raise instead of encoding something else."""
    import torch
    from d_kernels import F2, gen_arikan
    from polar.enc import PolarEncoder
    from polar.froze import get_Kern_frozen_bits
    assert F2.device.type == "cpu"                         # kernel matrices stay on the host (no CUDA context at import)
    G, _, fp = get_Kern_frozen_bits(64, 32, F2)
    assert PolarEncoder(fp, 64, G).G_ is None and PolarEncoder(fp, 64, None).k == 32
    bad = G.clone(); bad[5, 2] = 1
    for g in (bad, G.t().contiguous(), gen_arikan(torch.tensor([[1., 1.], [0., 1.]]), 6), G[:32, :32]):
        with pytest.raises(AssertionError):
            PolarEncoder(fp, 64, g)
