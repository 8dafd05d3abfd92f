"""GPU: the per-instance LV2 façade (lv2_descriptor / instantiate / connect_port / run / cleanup) of libb200meters.so
driven side by side with the REFERENCE plugins (oracle/_ref exports the reference's own lv2_descriptor: src/meters.cc
compiled unmodified), the way an LV2 host drives meters.so (robtk/jackwrap.c:531-544).  Every control-port value must
be bit-identical after every run(); cycles in which the reference emits rand()-based "force a parameter change"
values are compared by their sign/threshold only.  Without oracle/_ref the reference side is replayed from its recording
(tests/_reftape.py)."""
import ctypes as C

import numpy as np
import pytest

import _oracle as O
import _reftape as R
import _signals as S

pytestmark = pytest.mark.gpu
URI = b"http://gareus.org/oss/lv2/meters#"


class Desc(C.Structure):
    pass


class Feature(C.Structure):
    _fields_ = [("URI", C.c_char_p), ("data", C.c_void_p)]


MAPFN = C.CFUNCTYPE(C.c_uint32, C.c_void_p, C.c_char_p)


class UridMap(C.Structure):
    _fields_ = [("handle", C.c_void_p), ("map", MAPFN)]


Desc._fields_ = [("URI", C.c_char_p),
                 ("instantiate", C.CFUNCTYPE(C.c_void_p, C.POINTER(Desc), C.c_double, C.c_char_p, C.POINTER(C.POINTER(Feature)))),
                 ("connect_port", C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.c_void_p)),
                 ("activate", C.c_void_p),
                 ("run", C.CFUNCTYPE(None, C.c_void_p, C.c_uint32)),
                 ("deactivate", C.c_void_p),
                 ("cleanup", C.CFUNCTYPE(None, C.c_void_p)),
                 ("extension_data", C.c_void_p)]

_uris = {}


@MAPFN
def _map(handle, uri):
    """URID = 31 bits of the URI's CRC-32: the same number for a URI whatever was mapped before (recorded notify bytes and
    state blobs of the reference stay valid in any test order)"""
    import zlib
    u = zlib.crc32(uri) & 0x7FFFFFFF or 1
    assert _uris.setdefault(u, uri) == uri, (uri, _uris[u])
    return u


_urid_map = UridMap(None, _map)
_feat = Feature(b"http://lv2plug.in/ns/ext/urid#map", C.cast(C.pointer(_urid_map), C.c_void_p))
_feats = (C.POINTER(Feature) * 2)(C.pointer(_feat), None)


def descriptors(path):
    L = C.CDLL(path)
    L.lv2_descriptor.restype = C.POINTER(Desc); L.lv2_descriptor.argtypes = [C.c_uint32]
    out, i = {}, 0
    while True:
        d = L.lv2_descriptor(i)
        if not d:
            break
        out[d.contents.URI[len(URI):].decode()] = d
        i += 1
    return out, L


class Plugin:
    def __init__(self, d, rate=48000.0):
        self.d = d.contents
        self.h = self.d.instantiate(d, rate, b"", _feats)
        assert self.h
        self.keep = {}

    def port(self, idx, arr):
        self.keep[idx] = arr
        self.d.connect_port(self.h, idx, arr.ctypes.data_as(C.c_void_p))

    def run(self, n):
        self.d.run(self.h, n)

    def close(self):
        self.d.cleanup(self.h)


def u32(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _pair(name, t):
    import meters_lv2_b200 as B
    mine, l1 = descriptors(B.LIB_PATH)
    ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    return Plugin(mine[name]), t.obj(lambda: Plugin(ref[name])), (l1, l2)


def test_descriptor_table(reftape):
    import meters_lv2_b200 as B
    d, _ = descriptors(B.LIB_PATH)
    assert set(d) == {"COR", "spectr30mono", "spectr30stereo", "dBTPmono", "dBTPstereo", "K12mono", "K14mono", "K20mono",
                      "K12stereo", "K14stereo", "K20stereo", "TPnRMSmono", "TPnRMSstereo", "BBCM6", "EBUr128", "SigDistHist", "bitmeter", "dr14mono", "dr14stereo"} | {
                          k + c for k in ("VU", "BBC", "EBU", "DIN", "NOR") for c in ("mono", "stereo")} | {"surround%d" % k for k in range(3, 9)} | {"phasewheel", "stereoscope", "goniometer"}
    r = reftape.ref(lambda: sorted(descriptors(O.PATHS["reference"])[0]))
    assert set(d) == set(r) and len(r) == 38          # src/meters.cc:745-792


def _run_needle_family(t, name, ctl_ports, nch, script):
    """ports 0..9 layout of src/meters.cc:59-70; `script` maps block index -> value written to port 0 (ref level)"""
    g, r, keep = _pair(name, t)
    x = S.white(2, 1024 * 24, seed=91)
    gp = {i: np.zeros(1, np.float32) for i in ctl_ports}; rp = {i: np.zeros(1, np.float32) for i in ctl_ports}
    for i in ctl_ports:
        g.port(i, gp[i]); r.port(i, rp[i])
    for b in range(24):
        if b in script:
            gp[0][0] = rp[0][0] = script[b]
        bufs = [np.ascontiguousarray(x[c, b * 1024:(b + 1) * 1024]) for c in range(2)]
        for p, cp in ((g, gp), (r, rp)):
            mine = [a.copy() for a in bufs]
            p.port(1, mine[0]); p.port(2, mine[0])
            if nch == 2:
                p.port(4, mine[1]); p.port(5, mine[1])
            p.run(1024)
        rv = t.ref(lambda: [rp[i][0] for i in ctl_ports[1:]])
        for i, bb in zip(ctl_ports[1:], rv):
            a = gp[i][0]
            if bb <= -1.0 and (bb != np.floor(bb) or bb < -1.5):       # rand()-based forced change: same regime only
                assert a <= -1.0, (name, b, i, a, bb)
            else:
                assert u32(gp[i])[0] == u32(bb)[0], (name, b, i, a, bb)
    g.close(); r.close()


def test_kmeter_and_dbtp_plugins_vs_reference_plugins(reftape):
    script = {12: 1.0, 13: 3.0, 14: 4.0, 18: -3.0, 19: 0.5}              # peak-reset handshake values on port 0
    _run_needle_family(reftape, "K20stereo", [0, 3, 6, 7, 8, 9], 2, script)
    _run_needle_family(reftape, "K14stereo", [0, 3, 6, 7, 8, 9], 2, {})
    _run_needle_family(reftape, "dBTPstereo", [0, 3, 6, 7, 8], 2, script)
    _run_needle_family(reftape, "K20mono", [0, 3, 4, 5], 1, script)                 # mono: ports 4, 5 re-used for peak / hold
    _run_needle_family(reftape, "dBTPmono", [0, 3, 4], 1, script)


@pytest.mark.parametrize("name", ["VUstereo", "BBCstereo", "EBUmono", "DINstereo", "NORmono", "BBCM6"])
def test_needle_plugins_vs_reference_plugins(name, reftape):
    g, r, keep = _pair(name, reftape)
    x = S.white(2, 1024 * 14, seed=95) * np.float32(2.0)
    nch = 1 if name.endswith("mono") else 2
    cps = [0, 3, 6, 7]
    gp = {i: np.zeros(1, np.float32) for i in cps}; rp = {i: np.zeros(1, np.float32) for i in cps}
    for i in cps:
        g.port(i, gp[i]); r.port(i, rp[i])
    for b in range(14):
        if b == 5:
            gp[0][0] = rp[0][0] = -18.0                                      # reference level -> rlgain
        if b == 9:
            gp[7][0] = rp[7][0] = 1.0                                        # BBCM6: port 7 > 0.5 -> S meter +14 dB
        for p in (g, r):
            a = np.ascontiguousarray(x[0, b * 1024:(b + 1) * 1024]); c = np.ascontiguousarray(x[1, b * 1024:(b + 1) * 1024])
            p.port(1, a); p.port(2, a)
            if nch == 2:
                p.port(4, c); p.port(5, c)
            p.run(1024)
        r3, r6 = reftape.ref(lambda: [rp[3][0], rp[6][0]])
        assert u32(gp[3])[0] == u32(r3)[0], (name, b, gp[3][0], r3)
        if nch == 2:
            assert u32(gp[6])[0] == u32(r6)[0], (name, b, gp[6][0], r6)
    g.close(); r.close()


def test_cor_plugin_vs_reference_plugin(reftape):
    g, r, keep = _pair("COR", reftape)
    x = S.white(2, 1024 * 10, seed=93); x[1] = 0.5 * x[0] + 0.5 * x[1]
    gl, rl = np.zeros(1, np.float32), np.zeros(1, np.float32)
    g.port(3, gl); r.port(3, rl)
    for b in range(10):
        for p in (g, r):
            a = np.ascontiguousarray(x[0, b * 1024:(b + 1) * 1024]); c = np.ascontiguousarray(x[1, b * 1024:(b + 1) * 1024])
            o1, o2 = np.empty_like(a), np.empty_like(c)                     # out != in: pass-through copy
            p.port(1, a); p.port(2, o1); p.port(4, c); p.port(5, o2)
            p.run(1024)
            same = np.array_equal(o1, a) and np.array_equal(o2, c)
            assert same if p is g else reftape.ref(lambda: same)
        assert u32(gl)[0] == u32(reftape.ref(lambda: rl[0]))[0]
    g.close(); r.close()


def test_spectr30_plugin_vs_reference_plugin(reftape):
    g, r, keep = _pair("spectr30stereo", reftape)
    x = S.white(2, 1024 * 8, seed=92)
    outs = []
    for p in (g, r):
        out = np.zeros(60, np.float32); spd = np.ones(1, np.float32); rst = np.full(1, -4.0, np.float32); amp = np.zeros(1, np.float32)
        for i in range(60):
            p.d.connect_port(p.h, i, out[i:i + 1].ctypes.data_as(C.c_void_p))
        p.port(60, spd); p.port(61, rst); p.port(62, amp)
        outs.append((out, spd, rst))
    for b in range(8):
        if b == 4:
            for o in outs:
                o[1][0] = 3.0                                               # speed change: resets the peak hold (rst_h = 0)
        for p in (g, r):
            a = np.ascontiguousarray(x[0, b * 1024:(b + 1) * 1024]); c = np.ascontiguousarray(x[1, b * 1024:(b + 1) * 1024])
            p.port(64, a); p.port(65, a); p.port(66, c); p.port(67, c)
            p.run(1024)
        go, ro = outs[0][0], reftape.ref(lambda: outs[1][0])
        assert np.array_equal(u32(go[:30]), u32(ro[:30])), b
        pend = ro[30:] <= -500
        assert np.array_equal(pend, go[30:] <= -500) and np.array_equal(u32(go[30:][~pend]), u32(ro[30:][~pend])), b
    g.close(); r.close()


def test_tpnrms_plugin_vs_reference_plugin(reftape):
    g, r, keep = _pair("TPnRMSstereo", reftape)
    x = S.white(2, 1024 * 16, seed=94); x[0, 3000:3010] = 0.0
    ports = []
    seq = np.zeros(4, np.uint32)                                            # empty LV2 atom sequence: {size = 8, type, unit, pad}
    seq[0] = 8
    for p in (g, r):
        ctl = {i: np.zeros(1, np.float32) for i in (1, 2, 3, 6, 7, 8, 9, 10, 13, 14, 15, 16, 17, 18)}
        for i, a in ctl.items():
            p.port(i, a)
        p.port(0, seq)
        ports.append(ctl)
    for b in range(16):
        for ctl in ports:
            ctl[2][0] = 1.0 if b == 9 else 0.0                              # reset button
        for p in (g, r):
            a = np.ascontiguousarray(x[0, b * 1024:(b + 1) * 1024]); c = np.ascontiguousarray(x[1, b * 1024:(b + 1) * 1024])
            p.port(4, a); p.port(5, a); p.port(11, c); p.port(12, c)
            p.run(1024)
        outs = (3, 6, 7, 8, 9, 13, 14, 15, 16)
        for i, rv in zip(outs, reftape.ref(lambda: [ports[1][i][0] for i in outs])):
            assert u32(ports[0][i])[0] == u32(rv)[0], (b, i, ports[0][i][0], rv)
    g.close(); r.close()


@pytest.mark.parametrize("chn,pairs", [(5, [(0, 1), (2, 3), (0, 4), (9, 1)]), (3, [(0, 1), (1, 2), (2, 0)]), (8, [(7, 6), (5, 4), (3, 2), (1, 0)])])
def test_surround_meters_vs_reference_plugins(chn, pairs, reftape):
    """sur_run (src/surmeter.c:115-147): selectable-pair correlation meters (out-of-range selections clamp) + K-meters"""
    g, r, keep = _pair("surround%d" % chn, reftape)
    x = S.white(8, 1024 * 20, seed=97)
    x[1] = 0.6 * x[0] + 0.4 * x[1]; x[3] = -x[2]                           # correlated / anti-correlated pairs
    outs = []
    for p in (g, r):
        o = {}
        for c, (a, b) in enumerate(pairs):
            pa = np.full(1, a, np.float32); pb = np.full(1, b, np.float32); pc = np.zeros(1, np.float32)
            p.port(1 + 3 * c, pa); p.port(2 + 3 * c, pb); p.port(3 + 3 * c, pc); o[3 + 3 * c] = pc
        for c in range(chn):
            lv = np.zeros(1, np.float32); pk = np.zeros(1, np.float32)
            p.port(15 + 4 * c, lv); p.port(16 + 4 * c, pk); o[15 + 4 * c] = lv; o[16 + 4 * c] = pk
        p.port(0, np.zeros(1, np.float32))
        outs.append(o)
    for b in range(20):
        for p in (g, r):
            for c in range(chn):
                a = np.ascontiguousarray(x[c, b * 1024:(b + 1) * 1024])
                p.port(13 + 4 * c, a); p.port(14 + 4 * c, a)
            p.run(1024)
        for i, rv in zip(outs[0], reftape.ref(lambda: [outs[1][i][0] for i in outs[0]])):
            assert u32(outs[0][i])[0] == u32(rv)[0], (chn, b, i, outs[0][i][0], rv)
    g.close(); r.close()


@pytest.mark.parametrize("name,level_port", [("COR", 3), ("VUmono", 3), ("K20mono", 3)])
def test_audio_is_forwarded_whatever_the_cycle_length(name, level_port, reftape):
    """ADVICE r1: cycles longer than the engine's 8192-frame block are metered in pieces (the reference's needle / COR / K-meter
    plugins take any n, src/meters.cc:298-331,333-418,511-536) and the in -> out copy never depends on the metering."""
    g, r, keep = _pair(name, reftape)
    stereo = name == "COR"
    n = 8192 + 8192 + 1616
    x = S.white(2, n, seed=93)
    for p in (g, r):
        p.lvl = np.zeros(1, np.float32); p.refl = np.zeros(1, np.float32); p.aux = [np.zeros(1, np.float32) for _ in range(4)]
        p.outs = [np.full(n, 7.0, np.float32) for _ in range(2)]
        p.ins = [np.ascontiguousarray(x[c]) for c in range(2)]
        p.refl[0] = 20.0 if name[0] == "K" else -18.0          # K-meters: |port 0| < 3 is the GUI's re-init handshake (src/meters.cc:339-357)
        p.port(0, p.refl); p.port(1, p.ins[0]); p.port(2, p.outs[0]); p.port(level_port, p.lvl)
        if stereo:
            p.port(4, p.ins[1]); p.port(5, p.outs[1])
        else:
            p.port(4, p.aux[0]); p.port(5, p.aux[1])          # mono K-meter / VU: peak and hold live in the second channel's slots
        p.run(n)
    assert np.array_equal(g.outs[0], x[0]) and (not stereo or np.array_equal(g.outs[1], x[1]))
    assert np.isfinite(g.lvl[0]) and g.lvl[0] != 0
    # piecewise metering re-rounds a little (per-call scrubs / n mod 4 tails): the reading stays within the contract's 1e-4 dB
    rl = reftape.ref(lambda: r.lvl[0])
    assert abs(g.lvl[0] - rl) <= 1.2e-5 * abs(rl) + 1e-7, (g.lvl[0], rl)
    g.close(); r.close()


@pytest.mark.parametrize("name,ports,audio", [
    ("COR", [0, 3], [(1, 2), (4, 5)]),
    ("K20stereo", [0, 3, 6, 7, 8, 9], [(1, 2), (4, 5)]),
    ("dBTPmono", [0, 3, 4, 5], [(1, 2)]),
    ("VUstereo", [0, 3, 6], [(1, 2), (4, 5)]),
    ("DINmono", [0, 3], [(1, 2)]),
    ("spectr30stereo", list(range(64)), [(64, 65), (66, 67)]),
])
def test_batched_mode_of_the_control_port_plugins(name, ports, audio, monkeypatch, reftape):
    """B200M_LV2_BATCH: the instances of one plugin type share one bank (csrc/lv2_shim.cu ShimHub).  What an instance's control
    ports show after cycle k + 1 is bit for bit what the reference plugin shows after cycle k (one declared cycle of latency)."""
    import meters_lv2_b200 as B
    monkeypatch.setenv("B200M_LV2_BATCH", "8")
    n, nb, blk = 5, 30, 1024
    mine, l1 = descriptors(B.LIB_PATH)
    ref, l2 = reftape.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    gs = [Plugin(mine[name]) for _ in range(n)]; rs = [reftape.obj(lambda: Plugin(ref[name])) for _ in range(n)]
    x = S.white(2 * n, blk * nb, seed=97)
    x[2] *= 0.1; x[5] = x[4]
    spec = name.startswith("spectr30")
    gp = [{i: np.zeros(1, np.float32) for i in ports} for _ in range(n)]; rp = [{i: np.zeros(1, np.float32) for i in ports} for _ in range(n)]
    for plugs, pp in ((gs, gp), (rs, rp)):
        for k, p in enumerate(plugs):
            for i in ports:
                p.port(i, pp[k][i])
            if spec:
                pp[k][60][0] = 1.0; pp[k][61][0] = -4.0; pp[k][62][0] = 0.0
            else:
                pp[k][0][0] = 20.0 if name[0] == "K" or name.startswith("dBTP") else -18.0      # no re-init handshake (|port 0| >= 3)
    outs = [p for p in ports if p not in (0, 60, 61, 62, 63)]
    prev = [None] * n
    checked = 0
    for b in range(nb):
        for plugs, pp in ((gs, gp), (rs, rp)):
            for k, p in enumerate(plugs):
                bufs = [np.ascontiguousarray(x[2 * k + c, b * blk:(b + 1) * blk]) for c in range(len(audio))]
                for c, (pi, po) in enumerate(audio):
                    p.port(pi, bufs[c]); p.port(po, bufs[c])
                p.run(blk)
        for k in range(n):
            now_ref = dict(zip(outs, reftape.ref(lambda: [rp[k][i][0] for i in outs])))
            if prev[k] is not None and b >= 2:
                for i in outs:
                    a, r_ = gp[k][i][0], prev[k][i]
                    if spec and i >= 30 and r_ <= -500:
                        assert a <= -500                                   # rand()-based "force redraw" values (src/spectrumlv2.c:243-246)
                    else:
                        assert u32(np.float32(a))[()] == u32(np.float32(r_))[()], (name, b, k, i, a, r_)
                checked += 1
            prev[k] = now_ref
    assert checked >= n * (nb - 3)
    for p in gs + rs:
        p.close()
