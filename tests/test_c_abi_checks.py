"""Argument checks of every C entry point (include/polar_b200.h), on any machine.

Every call below is rejected -- or, with B == 0, accepted -- before the library makes a CUDA launch, so the test needs
no GPU.  The pointers are fake addresses that no call dereferences.  A row names the entry point, the one argument it
changes from a valid call, the return code and the `<who>:` prefix of polar_last_error()."""

D = 256                  # fake device / host address, 256-byte aligned
MIS = D + 4              # not 16-byte aligned
BIG = 1 << 40            # a workspace size no check rejects
NAN = float("nan")


def _callers(lib):
    """entry point -> a valid call on fake pointers (B = 5); keyword arguments replace one argument"""
    def sc(fn):
        return lambda n=64, B=5, lg=D, fm=D, up=D, ui=None, pos=None, k=32: fn(lg, fm, n, B, up, ui, pos, k, None)

    def scl(fn):
        return lambda n=64, L=8, B=5, lg=D, fm=D, best=D, ui=None, pos=None, k=32, crc=None, crc_len=0: fn(
            lg, fm, n, L, B, best, ui, pos, k, None, None, crc, crc_len, D, BIG, None)

    def hybrid(mode):
        return lambda n=64, L=8, B=5, lg=D, fm=D, best=D, ui=None, pos=None, k=32, crc=D, crc_len=6, mode=mode, ws=D, \
            wsb=BIG: lib.polar_scl_decode_hybrid(lg, fm, n, L, B, best, ui, pos, k, crc, crc_len, mode, None, ws, wsb, None)

    def belief(mode):
        return lambda n=64, B=5, T=20, mode=mode, lg=D, fm=D, up=D, ui=None, sl=None, pos=None, k=32: \
            lib.polar_belief_decode_f32(lg, fm, n, B, T, mode, up, ui, sl, pos, k, None)

    return {
        "sc": sc(lib.polar_sc_decode_f32),
        "sc_boxplus": sc(lib.polar_sc_decode_boxplus_f32),
        "scl": scl(lib.polar_scl_decode),
        "scl_boxplus": scl(lib.polar_scl_decode_boxplus),
        "scl_boxplus_pruned": scl(lib.polar_scl_decode_boxplus_pruned),
        "hybrid0": hybrid(0), "hybrid1": hybrid(1), "hybrid2": hybrid(2),
        "belief0": belief(0), "belief1": belief(1),
        "encode_packed": lambda n=64, B=5, u=D, c=D: lib.polar_encode_packed(u, n, B, c, None),
        "encode_f32": lambda n=64, k=32, B=5, u=D, rank=D, c=D: lib.polar_encode_f32(u, rank, n, k, B, c, None, None),
        "pack": lambda n=64, B=5, x=D, p=D: lib.polar_pack_bits_f32(x, n, B, p, None),
        "unpack": lambda n=64, k=32, B=5, p=D, pos=D, out=D: lib.polar_unpack_info_f32(p, pos, n, k, B, out, None),
        "gather": lambda nin=64, nout=48, B=5, x=D, idx=D, out=D: lib.polar_gather_cols_f32(x, idx, nin, nout, B, out, None),
        "rate_recover": lambda nin=48, nout=64, B=5, x=D, s0=D, s1=D, fill=D, out=D: lib.polar_rate_recover_f32(
            x, s0, s1, fill, nin, nout, B, out, None),
        "frontend": lambda n=64, B=5, no=0.5, fm=D, u=D, lg=D: lib.polar_awgn_frontend(1, 0, no, fm, n, B, u, None, lg, None),
        "nr5g_frontend": lambda n=128, e=128, crc_len=11, B=5, no=0.5, pm=D, rows=D, pos=D, idx=D, u=D, lg=D:
            lib.polar_nr5g_awgn_frontend(1, 0, no, pm, rows, pos, crc_len, idx, n, e, B, u, None, lg, None),
        "qpsk_awgn_llr": lambda n=64, B=5, no=0.5, c=D, lg=D: lib.polar_qpsk_awgn_llr(1, 0, no, c, n, B, lg, None),
        "bec_frontend": lambda n=64, B=5, pe=0.1, lmax=20.0, fm=D, u=D, lg=D: lib.polar_bec_frontend(
            1, 0, pe, lmax, fm, n, B, u, None, lg, None),
        "bec_llr": lambda n=64, B=5, pe=0.1, lmax=20.0, c=D, lg=D: lib.polar_bec_llr(1, 0, pe, lmax, c, n, B, lg, None),
        "count_packed": lambda n=64, B=5, a=D, b=D, cnt=D: lib.polar_count_errors_packed(a, b, None, n, B, cnt, None),
        "count_f32": lambda k=32, B=5, b=D, bh=D, cnt=D: lib.polar_count_errors_f32(b, bh, k, B, cnt, None),
        "osd": lambda n=8, k=4, t=1, B=2, lg=D, gm=D, cf=D: lib.polar_osd_decode(lg, gm, n, k, t, B, None, cf, None, None),
    }


# (entry point, changed arguments, code name, who); the rows of the SC, SCL, hybrid and BP decoders run for every arithmetic
_SC = [(dict(n=1), "EINVAL"), (dict(n=24), "EINVAL"), (dict(n=16384), "EINVAL"), (dict(B=-1), "EINVAL"),
       (dict(lg=None), "EINVAL"), (dict(fm=None), "EINVAL"), (dict(up=None), "EINVAL"), (dict(ui=D), "EINVAL"),
       (dict(ui=D, pos=D, k=-1), "EINVAL"), (dict(ui=D, pos=D, k=65), "EINVAL"), (dict(lg=MIS), "EALIGN")]
_SCL = [(dict(n=1), "EINVAL"), (dict(n=24), "EINVAL"), (dict(n=8192), "EINVAL"), (dict(L=0), "EINVAL"),
        (dict(L=3), "EINVAL"), (dict(L=64), "EINVAL"), (dict(B=-1), "EINVAL"), (dict(lg=None), "EINVAL"),
        (dict(fm=None), "EINVAL"), (dict(best=None), "EINVAL"), (dict(ui=D), "EINVAL"),
        (dict(ui=D, pos=D, k=65), "EINVAL"), (dict(crc_len=-1), "EINVAL"), (dict(crc_len=33), "EINVAL"),
        (dict(crc_len=6), "EINVAL"), (dict(crc=D, crc_len=6, k=0), "EINVAL"), (dict(crc=D, crc_len=6, k=65), "EINVAL")]
_HYBRID = [(dict(mode=3), "EINVAL", "hybrid"), (dict(mode=-1), "EINVAL", "hybrid"), (dict(B=1 << 31), "EINVAL", "hybrid"),
           (dict(n=24), "EINVAL", "hybrid"), (dict(n=8192), "EINVAL", "hybrid"), (dict(L=3), "EINVAL", "hybrid"),
           (dict(B=-1), "EINVAL", "hybrid"), (dict(crc_len=0), "EINVAL", "hybrid"), (dict(crc_len=33), "EINVAL", "hybrid"),
           (dict(crc=None), "EINVAL", "hybrid"), (dict(k=0), "EINVAL", "hybrid"), (dict(k=65), "EINVAL", "hybrid"),
           (dict(lg=None), "EINVAL", "hybrid"), (dict(fm=None), "EINVAL", "hybrid"), (dict(best=None), "EINVAL", "hybrid"),
           (dict(ui=D), "EINVAL", "hybrid"), (dict(ws=None), "ENOMEM", "hybrid"), (dict(wsb=1), "ENOMEM", "hybrid"),
           (dict(ws=D + 8), "EALIGN", "hybrid"),
           (dict(lg=MIS), "EALIGN", "sc")]          # the SC stage checks the rows
_BELIEF = [(dict(n=1), "EINVAL"), (dict(n=48), "EINVAL"), (dict(n=2048), "EINVAL"), (dict(T=0), "EINVAL"),
           (dict(mode=2), "EINVAL"), (dict(mode=-1), "EINVAL"), (dict(B=-1), "EINVAL"), (dict(lg=None), "EINVAL"),
           (dict(fm=None), "EINVAL"), (dict(up=None), "EINVAL"), (dict(ui=D), "EINVAL"), (dict(sl=D, pos=D, k=65), "EINVAL"),
           (dict(lg=MIS), "EALIGN")]
ROWS = ([(e, kw, rc, "sc") for e in ("sc", "sc_boxplus") for kw, rc in _SC]
        + [(e, kw, rc, "scl") for e in ("scl", "scl_boxplus", "scl_boxplus_pruned") for kw, rc in _SCL]
        + [("hybrid%d" % m, kw, rc, who) for m in range(3) for kw, rc, who in _HYBRID]
        + [("belief%d" % m, kw, rc, "belief") for m in range(2) for kw, rc in _BELIEF]
        + [("encode_packed", kw, "EINVAL", "encode") for kw in (dict(n=24), dict(n=16384), dict(B=-1), dict(u=None),
                                                                 dict(c=None))]
        + [("encode_f32", kw, "EINVAL", "encode") for kw in (dict(n=24), dict(B=-1), dict(k=-1), dict(k=65), dict(u=None),
                                                              dict(rank=None), dict(c=None))]
        + [("pack", kw, "EINVAL", "pack") for kw in (dict(n=0), dict(n=33), dict(B=-1), dict(x=None), dict(p=None))]
        + [("unpack", kw, "EINVAL", "unpack") for kw in (dict(n=0), dict(k=-1), dict(B=-1), dict(p=None), dict(pos=None),
                                                          dict(out=None))]
        + [("gather", kw, "EINVAL", "gather") for kw in (dict(nin=0), dict(nout=0), dict(B=-1), dict(x=None), dict(idx=None),
                                                          dict(out=None))]
        + [("rate_recover", kw, "EINVAL", "rate_recover") for kw in (dict(nin=0), dict(nout=0), dict(B=-1), dict(x=None),
                                                                      dict(s0=None), dict(s1=None), dict(fill=None),
                                                                      dict(out=None))]
        + [("frontend", kw, rc, "frontend") for kw, rc in (
            (dict(n=24), "EINVAL"), (dict(n=16384), "EINVAL"), (dict(B=-1), "EINVAL"), (dict(no=0.0), "EINVAL"),
            (dict(no=NAN), "EINVAL"), (dict(fm=None), "EINVAL"), (dict(lg=None), "EINVAL"), (dict(lg=MIS), "EALIGN"))]
        + [("nr5g_frontend", kw, "EINVAL", "nr5g frontend") for kw in (
            dict(n=16), dict(n=48), dict(n=2048), dict(e=0), dict(e=8193), dict(crc_len=0), dict(crc_len=33), dict(B=-1),
            dict(no=0.0), dict(pm=None), dict(rows=None), dict(pos=None), dict(idx=None), dict(u=None), dict(lg=None))]
        + [("qpsk_awgn_llr", kw, rc, "qpsk_awgn") for kw, rc in (
            (dict(n=0), "EINVAL"), (dict(n=6), "EINVAL"), (dict(B=-1), "EINVAL"), (dict(no=0.0), "EINVAL"),
            (dict(c=None), "EINVAL"), (dict(lg=None), "EINVAL"), (dict(c=MIS), "EALIGN"), (dict(lg=MIS), "EALIGN"))]
        + [("bec_frontend", kw, rc, "bec frontend") for kw, rc in (
            (dict(n=24), "EINVAL"), (dict(B=-1), "EINVAL"), (dict(pe=-0.1), "EINVAL"), (dict(pe=1.5), "EINVAL"),
            (dict(lmax=-1.0), "EINVAL"), (dict(fm=None), "EINVAL"), (dict(lg=None), "EINVAL"), (dict(lg=MIS), "EALIGN"))]
        + [("bec_llr", kw, rc, "bec") for kw, rc in (
            (dict(n=6), "EINVAL"), (dict(B=-1), "EINVAL"), (dict(pe=2.0), "EINVAL"), (dict(c=None), "EINVAL"),
            (dict(lg=None), "EINVAL"), (dict(c=MIS), "EALIGN"), (dict(lg=MIS), "EALIGN"))]
        + [("count_packed", kw, "EINVAL", "count") for kw in (dict(n=0), dict(B=-1), dict(a=None), dict(b=None),
                                                               dict(cnt=None))]
        + [("count_f32", kw, "EINVAL", "count") for kw in (dict(k=0), dict(B=-1), dict(b=None), dict(bh=None),
                                                            dict(cnt=None))]
        + [("osd", kw, "EINVAL", "osd") for kw in (dict(lg=None), dict(gm=None), dict(cf=None), dict(n=1), dict(n=1025),
                                                    dict(k=0), dict(k=9), dict(t=-1), dict(t=7), dict(B=-1),
                                                    dict(n=1024, k=512, t=6))])


def _code(dk, name):
    return getattr(dk, "POLAR_" + name)


def test_bad_device_calls_fail_before_any_launch():
    import d_kernels as dk
    lib = dk.lib()
    calls = _callers(lib)
    before = lib.polar_launch_count()
    for entry, kw, rc, who in ROWS:
        got = calls[entry](**kw)
        msg = lib.polar_last_error()
        assert got == _code(dk, rc), (entry, kw, got, msg)
        assert msg.startswith(who.encode() + b":"), (entry, kw, msg)
    assert lib.polar_launch_count() == before


def test_bad_host_and_setup_calls():
    import d_kernels as dk
    lib = dk.lib()
    sc_host = lambda n=64, B=5, lg=D, fm=D, up=D, ui=None, pos=None, k=32, dev=0: lib.polar_sc_decode_host_f32(
        lg, fm, n, B, up, ui, pos, k, dev)
    scl_host = lambda n=64, L=8, B=5, lg=D, fm=D, best=D, ui=None, pos=None, k=32, dev=0: lib.polar_scl_decode_host_f32(
        lg, fm, n, L, B, best, ui, pos, k, None, None, 0, dev)
    rows = ([(sc_host, kw, "sc host") for kw in (
                dict(n=1), dict(n=24), dict(n=16384), dict(B=-1), dict(lg=None), dict(fm=None), dict(up=None), dict(ui=D),
                dict(ui=D, pos=D, k=0), dict(ui=D, pos=D, k=65), dict(dev=-1), dict(dev=64))]
            + [(scl_host, kw, "scl host") for kw in (
                dict(n=24), dict(n=8192), dict(L=3), dict(B=-1), dict(lg=None), dict(fm=None), dict(best=None), dict(ui=D),
                dict(ui=D, pos=D, k=0), dict(dev=-1), dict(dev=64))]
            + [(lambda: lib.polar_sc_decode_host(D, D, 64, 5, None, 0), {}, "sc host"),
               (lambda: lib.polar_scl_decode_host(D, D, 64, 8, 5, None, None, None, 0, 0), {}, "scl host"),
               (lambda: lib.polar_mc_control_group(None, D, 1, D, 1, D, 0, -1, -1, 1, 0, None), {}, "mc_control_group"),
               (lambda: lib.polar_mc_control_group(D, D, 0, D, 1, D, 0, -1, -1, 1, 0, None), {}, "mc_control_group"),
               (lambda: lib.polar_mc_control_group(D, D, 33, D, 1, D, 0, -1, -1, 1, 0, None), {}, "mc_control_group"),
               (lambda: lib.polar_mc_control_group(D, D, 1, D, 1, D, 0, -1, -1, 0, 0, None), {}, "mc_control_group"),
               (lambda: lib.polar_scl3_math_selftest(1, None, None), {}, "selftest"),
               (lambda: lib.polar_init(-1), {}, "init"),
               (lambda: lib.polar_set_option(b"NOT_POLAR", 1), {}, "set_option")])
    before = lib.polar_launch_count()
    for fn, kw, who in rows:
        got = fn(**kw)
        msg = lib.polar_last_error()
        assert got == dk.POLAR_EINVAL, (who, kw, got, msg)
        assert msg.startswith(who.encode() + b":"), (who, kw, msg)
    assert lib.polar_launch_count() == before
    assert lib.polar_sc_decode_host_f32(None, None, 64, 0, None, None, None, 0, 0) == dk.POLAR_OK
    assert lib.polar_scl_decode_host_f32(None, None, 64, 8, 0, None, None, None, 0, None, None, 0, 0) == dk.POLAR_OK


def test_empty_batch_launches_nothing():
    import d_kernels as dk
    lib = dk.lib()
    calls = _callers(lib)
    assert set(calls) >= {"sc", "sc_boxplus", "scl", "scl_boxplus", "scl_boxplus_pruned", "hybrid0", "hybrid1", "hybrid2",
                          "belief0", "belief1"}
    before = lib.polar_launch_count()
    for entry, call in calls.items():
        assert call(B=0) == dk.POLAR_OK, (entry, lib.polar_last_error())
    assert calls["sc"](B=0, lg=None, fm=None, up=None) == dk.POLAR_OK            # B == 0 passes whatever its buffers
    assert calls["scl"](B=0, lg=None, fm=None, best=None) == dk.POLAR_OK
    assert calls["belief1"](B=0, n=1024, lg=None, fm=None, up=None) == dk.POLAR_OK
    assert calls["unpack"](k=0) == dk.POLAR_OK                                   # no information bits: nothing to do
    assert lib.polar_launch_count() == before
    for ws_bytes in (lib.polar_scl_workspace_bytes, lib.polar_scl_boxplus_workspace_bytes):
        assert ws_bytes(64, 8, 0) == 0 and ws_bytes(24, 8, 5) == 0 and ws_bytes(64, 3, 5) == 0
    for mode in range(3):
        assert lib.polar_scl_hybrid_workspace_bytes(64, 8, 0, mode) == 0
    assert lib.polar_scl_hybrid_workspace_bytes(64, 8, 5, 3) == 0
