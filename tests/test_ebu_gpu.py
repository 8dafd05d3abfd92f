"""GPU parity: b200m_ebu_* (CUDA) vs the CPU oracle, same seeded inputs, same block sequence."""
import numpy as np
import pytest

import _oracle as O
import _signals as S

pytestmark = pytest.mark.gpu
RES = ("loudness_M", "maxloudn_M", "loudness_S", "maxloudn_S", "integrated", "integ_thr", "range_min", "range_max", "range_thr")


def _run_both(x, blocks, nchan=2, start=True, host=False, check_state=True):
    """x: [C, total] ; blocks: list of block lengths.  Returns (gpu results, oracle results)."""
    import torch
    import meters_lv2_b200 as B
    C = x.shape[0]
    n_inst = C // nchan
    g = B.Ebu_r128_proc(n_inst, nchan)
    o = O.Ebu(n_inst, nchan)
    if start:
        g.integr_start(); o.integr("start")
    xd = None if host else torch.from_numpy(x).cuda()
    pos = 0
    for n in blocks:
        blk = np.ascontiguousarray(x[:, pos:pos + n])
        o.process(blk, nthreads=8)
        if host:
            g.process(blk)
        else:
            g.process(xd[:, pos:pos + n])
        pos += n
    gr = g.results()
    orr = o.read()
    return g, o, gr, orr


def _assert_equal(g, o, gr, orr, n_inst, nchan=2, exact=True):
    for i, name in enumerate(RES):
        a, b = gr[name], orr[:, i]
        if exact:
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (name, a[:4], b[:4], int((a != b).sum()))
        else:
            assert np.allclose(a, b, atol=1e-4, rtol=0), name      # +-1e-4 dB (north_star tolerance)
    for inst in sorted(set([0, n_inst // 2, n_inst - 1])):
        hm, hs = g.histogram(inst)
        om, os_, oc = o.hist(inst)
        assert np.array_equal(hm, om) and np.array_equal(hs, os_), "histogram counts must be bit-exact"
        assert gr["hist_M_count"][inst] == oc[0] and gr["hist_S_count"][inst] == oc[1]
        z, pw, fr, c = g.state(inst)
        oz, opw, ofr, oc4 = o.state(inst)
        assert np.array_equal(z.view(np.uint32), oz.view(np.uint32)), "filter state"
        assert np.array_equal(pw.view(np.uint32), opw.view(np.uint32)), "fragment power ring"
        assert np.float32(fr).view(np.uint32) == np.float32(ofr).view(np.uint32)
        assert list(c) == list(oc4)


def test_coeffs_bitwise():
    import meters_lv2_b200 as B
    for fs in (48000.0, 44100.0, 96000.0):
        g = B.Ebu_r128_proc(1, 2, fs)
        o = O.Ebu(1, 2, fs)
        assert np.array_equal(g.coeffs().view(np.uint32), o.coeffs().view(np.uint32))


@pytest.mark.parametrize("n_inst,blocks", [
    (37, [1024] * 60),                        # ~1.3 s : M, S live, I not yet (count < 50)
    (64, [1024] * 300),                       # 6.4 s : integrated loudness + LRA gate live
    (5, [64] * 100 + [480] * 40 + [8192] * 6 + [1, 3, 7, 1023, 2401, 4799]),   # ragged sequence
])
def test_white_noise_bit_exact(n_inst, blocks):
    x = S.white(2 * n_inst, sum(blocks))
    g, o, gr, orr = _run_both(x, blocks)
    _assert_equal(g, o, gr, orr, n_inst)


@pytest.mark.parametrize("env", ["B200M_EBU_TMA=1", "B200M_EBU_SPLIT=1"])
def test_alternative_k1_kernels_are_bit_identical(monkeypatch, env):
    """the K-weighting kernel exists in three forms: one warp per 32 channels with cp.async staging (default), two warps per 32
    channels (B200M_EBU_SPLIT=1, ebu_kweight_split) and one warp with TMA staging (B200M_EBU_TMA=1: 128B-swizzled boxes, mbarrier).  All produce the
    same bits, incl. ragged blocks (partial tiles, fragment cuts inside a tile) and a mono bank"""
    monkeypatch.setenv(*env.split("="))
    blocks = [1024] * 40 + [64] * 30 + [480] * 20 + [8192] * 3 + [4, 8, 1020, 2404, 4800]
    x = S.white(2 * 37, sum(blocks), seed=31)
    g, o, gr, orr = _run_both(x, blocks)
    _assert_equal(g, o, gr, orr, 37)
    x1 = S.white(40, 1024 * 30, seed=32)
    g, o, gr, orr = _run_both(x1, [1024] * 30, nchan=1)
    _assert_equal(g, o, gr, orr, 40, nchan=1)


@pytest.mark.parametrize("nchan", [3, 4, 5])
def test_surround_banks(nchan):
    """Ebu_r128_proc::init (nchan = 3..5): channel gains 1 1 1 1.41 1.41 summed in channel order (ebu_r128_proc.cc:29,328-329);
    instances do not align with warps (30 of 32 lanes busy for 3 and 5 channels), ragged blocks, host path"""
    n_inst = 45
    blocks = [1024] * 118 + [480, 4800, 8192, 7, 64, 2401]
    x = S.white(n_inst * nchan, sum(blocks), seed=40 + nchan)
    g, o, gr, orr = _run_both(x, blocks, nchan=nchan)
    _assert_equal(g, o, gr, orr, n_inst, nchan=nchan)
    g, o, gr, orr = _run_both(x[:, :1000 * 20 + 1][:, 1:], [1000] * 20, nchan=nchan, host=True)       # unaligned rows through the host path
    _assert_equal(g, o, gr, orr, n_inst, nchan=nchan)


def test_mono_bank():
    x = S.white(33, 1024 * 120)
    g, o, gr, orr = _run_both(x, [1024] * 120, nchan=1)
    _assert_equal(g, o, gr, orr, 33, nchan=1)


def test_host_path_and_unaligned_stride():
    x = S.white(2 * 9, 1000 * 130 + 3)[:, 3:]              # rows start 12 bytes off a 16-byte boundary
    x = x[:, :1000 * 130]
    assert not x.flags.c_contiguous
    import meters_lv2_b200 as B
    g = B.Ebu_r128_proc(9, 2); o = O.Ebu(9, 2)
    g.integr_start(); o.integr("start")
    for b in range(130):
        blk = x[:, b * 1000:(b + 1) * 1000]
        g.process(blk)                                      # host path (numpy view, odd stride)
        o.process(np.ascontiguousarray(blk))
    _assert_equal(g, o, g.results(), o.read(), 9)


def test_nan_inf_denormal_scrub():
    x = S.nasty(2 * 8, 1024 * 64)
    g, o, gr, orr = _run_both(x, [1024] * 64)
    for i, name in enumerate(RES):
        a, b = gr[name], orr[:, i]
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), name
    z, pw, fr, c = g.state(3); oz, opw, ofr, oc4 = o.state(3)
    assert np.array_equal(z.view(np.uint32), oz.view(np.uint32))


def test_ebu_tech3341_tone():
    # 997 Hz, -23 dBFS, L = R  =>  -23.0 LUFS (EBU Tech 3341 case 1); oracle gives M = -23.007 (SURVEY App. C)
    n = 1024 * 300                                       # 6.4 s: > 50 momentary points, so I is live
    s = S.sine(n, 997.0, amp=10 ** (-23 / 20))
    x = np.ascontiguousarray(np.stack([s, s]))
    g, o, gr, orr = _run_both(x, [1024] * 300)
    _assert_equal(g, o, gr, orr, 1)
    assert abs(gr["loudness_M"][0] + 23.0) < 0.02 and abs(gr["integrated"][0] + 23.0) < 0.2   # I still carries the start-up transient after 6.4 s


def test_integration_controls_and_pause():
    import torch
    import meters_lv2_b200 as B
    x = S.white(2 * 6, 1024 * 150)
    g = B.Ebu_r128_proc(6, 2); o = O.Ebu(6, 2)
    xd = torch.from_numpy(x).cuda()
    for b in range(150):
        if b == 10:
            g.integr_start(); o.integr("start")
        if b == 80:
            g.integr_pause(2); o.integr("pause", 2)
        if b == 100:
            g.integr_reset(4); o.integr("reset", 4)
        if b == 120:
            g.integr_start(2); o.integr("start", 2)
        g.process(xd[:, b * 1024:(b + 1) * 1024]); o.process(np.ascontiguousarray(x[:, b * 1024:(b + 1) * 1024]))
    _assert_equal(g, o, g.results(), o.read(), 6)


def test_whole_mix_histogram_extension():
    import torch
    import meters_lv2_b200 as B
    n_inst = 48
    x = S.white(2 * n_inst, 1024 * 260)
    g, o, gr, orr = _run_both(x, [1024] * 260)
    mix = torch.zeros(B.MIX_WORDS, dtype=torch.int32, device="cuda")
    g.mix_reduce(mix)
    m = mix.cpu().numpy()
    hm = np.zeros(751, np.int64); hs = np.zeros(751, np.int64); cm = cs = 0
    for i in range(n_inst):
        a, b, c = o.hist(i); hm += a; hs += b; cm += c[0]; cs += c[1]
    assert np.array_equal(m[:751], hm) and np.array_equal(m[752:752 + 751], hs) and m[1504] == cm and m[1505] == cs
    out = g.mix_finish(mix)
    assert np.isfinite(out).all() and -40 < out[0] < 0


def test_sharded_banks_equal_single_bank():
    """multi-GPU = replicas over disjoint instance ranges: two half banks (as two ranks would own them) must equal
    one full bank bit for bit, and their all-reduced mix vector must equal the full bank's."""
    import torch
    import meters_lv2_b200 as B
    from meters_lv2_b200 import shard
    n = 22
    x = S.white(2 * n, 1024 * 140, seed=66)
    xd = torch.from_numpy(x).cuda()
    full = B.Ebu_r128_proc(n, 2); full.integr_start()
    parts = []
    for r in range(2):
        lo, cnt = shard.shard_range(n, r, 2)
        b = B.Ebu_r128_proc(cnt, 2); b.integr_start(); parts.append((lo, cnt, b))
    for blk in range(140):
        v = xd[:, blk * 1024:(blk + 1) * 1024]
        full.process(v)
        for lo, cnt, b in parts:
            b.process(v[2 * lo:2 * (lo + cnt)])
    fr = full.results()
    cat = np.concatenate([b.results() for _, _, b in parts])
    assert np.array_equal(fr.view(np.uint8), cat.view(np.uint8))
    mf = torch.zeros(B.MIX_WORDS, dtype=torch.int32, device="cuda"); full.mix_reduce(mf)
    acc = torch.zeros_like(mf)
    for _, _, b in parts:
        m = torch.zeros_like(mf); b.mix_reduce(m); acc += m
    assert torch.equal(mf, acc)
    assert np.array_equal(full.mix_finish(mf).view(np.uint32), parts[0][2].mix_finish(acc).view(np.uint32))


def test_ebur128_plugin_cycle_with_dbtp():
    """b200m_r128_*: ebur128_run's audio cycle (src/ebulv2.cc:341-367), device and host paths."""
    import torch
    import meters_lv2_b200 as B
    n = 12
    x = S.white(2 * n, 1024 * 130, seed=67)
    xd = torch.from_numpy(x).cuda()
    for host in (False, True):
        g = B.EBUr128(n, 48000.0, True); g.control(B.EBUr128.START)
        oe = O.Ebu(n, 2); ot = O.TruePeak(2 * n); oe.integr("start")
        tpmax = np.full(n, -np.inf, np.float32)
        for b in range(130):
            blk = np.ascontiguousarray(x[:, b * 1024:(b + 1) * 1024])
            g.run(blk if host else xd[:, b * 1024:(b + 1) * 1024])
            oe.process(blk); ot.process(blk, mode=1)
            m, _ = ot.read()
            v = np.maximum(m[0::2], m[1::2])
            tp = np.float32(20.0) * np.log10(v)            # compared with 1e-4 dB tolerance below, exact on device
            tpmax = np.maximum(tpmax, tp.astype(np.float32))
        res, tp = g.results()
        orr = o_read = oe.read()
        for i, name in enumerate(RES):
            assert np.array_equal(res[name].view(np.uint32), orr[:, i].view(np.uint32)), name
        assert np.abs(tp - tpmax).max() < 1e-4
    g2 = B.EBUr128(3, 48000.0, False)
    g2.run(xd[:6, :1024])
    assert np.isneginf(g2.results()[1]).all()              # dBTP disabled: tp_max = -inf (:365-366)


def test_r128_bank_vs_reference_ebur128_plugin(reftape):
    """b200m_r128_* against the reference's EBUr128 PLUGIN driven through its own ebur128_run (oracle/_ref compiles
    src/meters.cc unmodified): the nine loudness values and the dBTP hold tp_max must be bit-identical."""
    import torch
    import meters_lv2_b200 as B
    n = 10
    x = S.white(2 * n, 1024 * 140, seed=68)
    x[3] = 0
    xd = torch.from_numpy(x).cuda()
    g = B.EBUr128(n, 48000.0, True); g.control(B.EBUr128.START)
    o = reftape.obj(lambda: O.EbuPlugin(n, 48000.0, True))                # replayed from tests/golden/ref without oracle/_ref
    for b in range(140):
        g.run(xd[:, b * 1024:(b + 1) * 1024]); o.run(np.ascontiguousarray(x[:, b * 1024:(b + 1) * 1024]), nthreads=8)
        if b % 20 == 19:
            res, tp = g.results(); ref = reftape.ref(lambda: o.read())
            for i, name in enumerate(RES):
                assert np.array_equal(res[name].view(np.uint32), ref[:, i].view(np.uint32)), (b, name)
            assert np.array_equal(tp.view(np.uint32), ref[:, 9].view(np.uint32)), (b, tp, ref[:, 9])


def test_r128_snapshot_restore_continues_bit_identically():
    """checkpoint / resume: a fresh bank restored from a snapshot continues exactly like the original (results, tp_max,
    histograms), including the host-tracked fragment clock and gating phases (blocks of 1000 frames: the 2400-frame
    fragment boundary falls at a different offset in every block)."""
    import torch
    import meters_lv2_b200 as B
    n, blk, nb1, nb2 = 9, 1000, 37, 55
    x = S.white(2 * n, blk * (nb1 + nb2), seed=77)
    xd = torch.from_numpy(x).cuda()
    a = B.EBUr128(n, 48000.0, dbtp_enable=True); a.control(B.EBUr128.START)
    for b in range(nb1):
        if b == 20:
            a.control(B.EBUr128.PAUSE, 3)                    # per-instance control state must travel too
        a.run(xd[:, b * blk:(b + 1) * blk])
    blob = a.snapshot()
    c = B.EBUr128(n, 48000.0, dbtp_enable=False)             # dbtp flag comes from the snapshot
    c.restore(blob)
    for b in range(nb1, nb1 + nb2):
        if b == nb1 + 10:
            a.control(B.EBUr128.START, 3); c.control(B.EBUr128.START, 3)
        a.run(xd[:, b * blk:(b + 1) * blk]); c.run(xd[:, b * blk:(b + 1) * blk])
    ra, ta = a.results(); rc, tc = c.results()
    assert ra.tobytes() == rc.tobytes() and ta.tobytes() == tc.tobytes()
    for inst in (0, 3, n - 1):
        ma, sa = a.histogram(inst); mc, sc = c.histogram(inst)
        assert np.array_equal(ma, mc) and np.array_equal(sa, sc) and ma.sum() > 0
    with pytest.raises(Exception):
        B.EBUr128(n + 1, 48000.0).restore(blob)             # shape mismatch is refused
