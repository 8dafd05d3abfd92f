"""GPU: the goniometer plugin of the LV2 façade (csrc/lv2_gon.cu) side by side with the reference's (src/goniometerlv2.c:44-330,
compiled unmodified into oracle/_ref).  The reference GUI reaches the plugin through LV2 instance-access: it casts the instance
handle to `LV2gm*` (src/goniometer.h:113-169) and reads the ring buffer / flips `ui_active` in it.  The test does exactly that to
BOTH handles, at the offsets the two libraries report for their own structs (which must agree).  Without oracle/_ref the
reference side is replayed from its recording (tests/_reftape.py)."""
import ctypes as C

import numpy as np
import pytest

import _oracle as O
import _reftape as R
import _signals as S
from test_lv2_shim_gpu import Plugin, descriptors, u32

pytestmark = pytest.mark.gpu
FIELDS = ("rb", "ui_active", "rb_overrun", "s_sfact", "s_linewidth", "input", "rate", "ntfy", "msg_thread_lock", "map", "sizeof")


def _ref_layout():
    b = (C.c_size_t * 16)()
    m = C.CDLL(O.PATHS["reference"]).refgon_layout(b, 16)
    return list(b)[:m]


def _layouts(t):
    import meters_lv2_b200 as B
    a = (C.c_size_t * 16)()
    n = C.CDLL(B.LIB_PATH).b200m_lv2_gon_layout(a, 16)
    return dict(zip(FIELDS, list(a)[:n])), dict(zip(FIELDS, (int(v) for v in t.ref(_ref_layout))))


class Ring(C.Structure):                                   # gmringbuf, src/goniometer.h:33-39
    _fields_ = [("c0", C.POINTER(C.c_float)), ("c1", C.POINTER(C.c_float)), ("rp", C.c_size_t), ("wp", C.c_size_t), ("len", C.c_size_t)]


def _ring(handle, off):
    return C.cast(C.c_void_p.from_address(handle + off["rb"]).value, C.POINTER(Ring)).contents


def test_instance_struct_layout_matches_the_reference(reftape):
    mine, ref = _layouts(reftape)
    assert mine == ref and mine["sizeof"] == 208


def _ring_state(p, rb, off):
    """write / read position, rb_overrun and ntfy of a goniometer instance"""
    return [rb.wp, rb.rp, int(C.c_bool.from_address(p.h + off["rb_overrun"]).value), C.c_uint32.from_address(p.h + off["ntfy"]).value]


def test_goniometer_feed_and_correlation(reftape):
    import meters_lv2_b200 as B
    t = reftape
    off, _ = _layouts(t)
    mine, l1 = descriptors(B.LIB_PATH); ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    assert "goniometer" in mine and len(mine) == 38 == t.ref(lambda: len(ref))
    g, r = Plugin(mine["goniometer"]), t.obj(lambda: Plugin(ref["goniometer"]))
    live = (g, r) if t.live else (g,)                       # the instances whose memory this process can reach
    n, nb = 1024, 24
    x = S.white(2, n * nb, seed=71); x[1, : n * 6] = x[0, : n * 6]
    for p in (g, r):
        p.gain = np.ones(1, np.float32); p.corr = np.full(1, 9.0, np.float32); p.ntf = np.full(1, -1.0, np.float32)
        p.port(4, p.gain); p.port(5, p.corr); p.port(6, p.ntf)
    rg, rr = _ring(g.h, off), t.obj(lambda: _ring(r.h, off))
    rlen, rwp = t.ref(lambda: [rr.len, rr.wp])
    assert rg.len == rlen == 9600 and rg.wp == rwp == 0
    for b in range(nb):
        if b == 4:                                          # the GUI opens: ui_active = true through instance-access
            for p in live:
                C.c_bool.from_address(p.h + off["ui_active"]).value = True
        if b == 12:                                         # the GUI drains the ring (gmrb_read_clear) and acknowledges the overrun
            for p, rb in zip(live, (rg, rr)):
                rb.rp = rb.wp
                C.c_bool.from_address(p.h + off["rb_overrun"]).value = False
        for p in (g, r):
            ins = [np.ascontiguousarray(x[c, b * n:(b + 1) * n]) for c in range(2)]
            outs = [np.zeros(n, np.float32) for _ in range(2)]
            p.port(0, ins[0]); p.port(1, outs[0]); p.port(2, ins[1]); p.port(3, outs[1])
            p.run(n)
            same = np.array_equal(outs[0], ins[0]) and np.array_equal(outs[1], ins[1])
            assert same if p is g else t.ref(lambda: same)
        rcorr, rntf = t.ref(lambda: [r.corr[0], r.ntf[0]])
        assert u32(g.corr)[0] == u32(rcorr)[0], (b, g.corr, rcorr)           # untouched (9.0) while the GUI is closed, cor->read () after
        assert g.ntf[0] == rntf
        assert _ring_state(g, rg, off) == list(t.ref(lambda: _ring_state(r, rr, off))), b
    for ch in ("c0", "c1"):
        a = np.ctypeslib.as_array(getattr(rg, ch), shape=(rg.len,))
        assert R.digest(a[:rg.wp]) == t.digest(lambda: np.ctypeslib.as_array(getattr(rr, ch), shape=(rr.len,))[:rr.wp])
    assert g.corr[0] != 9.0 and abs(g.corr[0]) <= 1.0
    g.close(); r.close()


def test_goniometer_state_save_restore(reftape):
    """LV2 state (src/goniometerlv2.c:209-294): two atom:Vector blobs; what one plugin saves the other restores identically"""
    import meters_lv2_b200 as B
    from test_lv2_shim_gpu import _map, _uris
    t = reftape
    off, _ = _layouts(t)
    mine, l1 = descriptors(B.LIB_PATH); ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    STORE = C.CFUNCTYPE(C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32)
    RETR = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_size_t), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32))

    class Iface(C.Structure):
        _fields_ = [("save", C.CFUNCTYPE(C.c_uint32, C.c_void_p, STORE, C.c_void_p, C.c_uint32, C.c_void_p)),
                    ("restore", C.CFUNCTYPE(C.c_uint32, C.c_void_p, RETR, C.c_void_p, C.c_uint32, C.c_void_p))]

    def save(lib_desc):
        p = Plugin(lib_desc["goniometer"])
        C.c_int.from_address(p.h + off["s_sfact"]).value = 8
        C.c_float.from_address(p.h + off["s_linewidth"]).value = 1.25
        C.c_bool.from_address(p.h + off["rb_overrun"] + 1).value = True           # s_autogain follows rb_overrun
        ext = C.CFUNCTYPE(C.c_void_p, C.c_char_p)(p.d.extension_data)(b"http://lv2plug.in/ns/ext/state#interface")
        iface = C.cast(ext, C.POINTER(Iface)).contents
        got = {}

        @STORE
        def store(handle, key, value, size, typ, flags):
            got[key] = (C.string_at(value, size), typ, flags)
            return 0
        iface.save(p.h, store, None, 0, None)
        p.close()
        return got

    blobs = {"mine": save(mine)}
    got = t.obj(lambda: save(ref))
    # the reference's blobs with their key and type URIDs as URIs, so that the recording does not depend on the URID map
    keys = t.ref(lambda: [[_uris[k], _uris[v[1]]] for k, v in sorted(got.items())])
    flags = t.ref(lambda: [v[2] for k, v in sorted(got.items())])
    blobs["ref"] = {_map(None, bytes(k)): (t.ref(lambda: np.frombuffer(got[_map(None, bytes(k))][0], np.uint8)).tobytes(), _map(None, bytes(ty)), int(f))
                    for (k, ty), f in zip(keys, flags)}
    assert blobs["mine"] == blobs["ref"] and len(blobs["mine"]) == 2
    # restore the reference's blobs into a fresh instance of ours
    p = Plugin(mine["goniometer"])
    ext = C.CFUNCTYPE(C.c_void_p, C.c_char_p)(p.d.extension_data)(b"http://lv2plug.in/ns/ext/state#interface")
    iface = C.cast(ext, C.POINTER(Iface)).contents
    keep = {}

    @RETR
    def retrieve(handle, key, size, typ, flags):
        if key not in blobs["ref"]:
            return None
        data, t, f = blobs["ref"][key]
        keep[key] = C.create_string_buffer(data, len(data))
        size[0] = len(data); typ[0] = t; flags[0] = f
        return C.addressof(keep[key])
    iface.restore(p.h, retrieve, None, 0, None)
    assert C.c_int.from_address(p.h + off["s_sfact"]).value == 8
    assert C.c_float.from_address(p.h + off["s_linewidth"]).value == 1.25
    assert C.c_bool.from_address(p.h + off["rb_overrun"] + 1).value is True
    p.close()
