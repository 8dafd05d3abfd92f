"""GPU: the EBUr128 LV2 plugin of libb200meters.so (csrc/lv2_ebur128.cu) against the REFERENCE plugin (src/ebulv2.cc
compiled unmodified into oracle/_ref, -DHAVE_LV2_1_8 as every LV2 >= 1.8.1 build defines), both driven like an LV2 host
drives them: the same URID map, the same control-port atom sequences (meteron, metercfg key/value, time:Position), the
same audio.  After every run() the notify-port buffers must be IDENTICAL BYTES: every radar point, histogram delta,
ebulevels float and control reply.  The atom wire format itself is restated from the LV2 specification on both sides
(the SDK is not installed; oracle/lv2stub is the stand-in the reference is compiled against).  Without oracle/_ref the
reference side is replayed from its recording (tests/_reftape.py): notify buffers by length and digest."""
import ctypes as C
import struct

import numpy as np
import pytest

import _oracle as O
import _reftape as R
import _signals as S
from test_lv2_shim_gpu import Feature, _map, descriptors, Plugin

pytestmark = pytest.mark.gpu
ATOM = b"http://lv2plug.in/ns/ext/atom#"
TIME = b"http://lv2plug.in/ns/ext/time#"
MTR = b"http://gareus.org/oss/lv2/meters#"
CTL = dict(START=1, PAUSE=2, RESET=3, TRANSPORTSYNC=4, AUTORESET=5, RADARTIME=6, UISETTINGS=7, WINDOWED=13, AVERAGE=14)   # src/uris.h:187-203
CAP = 8192


def urid(uri):
    return _map(None, uri)


def obj(otype, props=()):
    """one event at frame 0 holding an atom:Object {otype; (key, type, packed 4-byte value)...}"""
    body = struct.pack("<II", 0, urid(otype))
    for key, typ, val in props:
        body += struct.pack("<IIII", urid(key), 0, 4, urid(typ)) + val + b"\0\0\0\0"
    return struct.pack("<q", 0) + struct.pack("<II", len(body), urid(ATOM + b"Object")) + body


def cfg(key, value):
    return obj(MTR + b"metercfg", [(MTR + b"controlkey", ATOM + b"Int", struct.pack("<i", CTL[key])),
                                   (MTR + b"controlval", ATOM + b"Float", struct.pack("<f", value))])


def position(speed):
    return obj(TIME + b"Position", [(TIME + b"speed", ATOM + b"Float", struct.pack("<f", speed))])


def sequence(events):
    body = struct.pack("<II", 0, 0) + b"".join(events)
    raw = struct.pack("<II", len(body), urid(ATOM + b"Sequence")) + body
    a = np.zeros(max(64, (len(raw) + 7) // 8 * 8), np.uint8)
    a[:len(raw)] = np.frombuffer(raw, np.uint8)
    return a


def drive(t, script, nblocks, block=1024, x=None, cap=CAP, rate=48000.0, name="EBUr128", nch=2):
    """script: {block index: [events]} fed to the control port of both plugins; asserts byte parity of the notify port"""
    import meters_lv2_b200 as B
    mine, l1 = descriptors(B.LIB_PATH)
    ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    g, r = Plugin(mine[name], rate), t.obj(lambda: Plugin(ref[name], rate))
    if x is None:
        x = S.white(2, block * nblocks, seed=17) * np.float32(4.0)
    empty = sequence([])
    notes = [np.zeros(cap, np.uint8), np.zeros(cap, np.uint8)]
    sizes = []
    for b in range(nblocks):
        ctl = sequence(script[b]) if b in script else empty
        outs = []
        for p, note in ((g, notes[0]), (r, notes[1])):
            note[:] = 0xA5                                                # stale bytes must not leak into the comparison
            note[:8] = np.frombuffer(struct.pack("<II", cap - 8, 0), np.uint8)   # host convention: capacity, type 0
            bufs = [np.ascontiguousarray(x[c, b * block:(b + 1) * block]) for c in range(nch)]
            p.port(0, ctl); p.port(1, note)
            for c in range(nch):
                p.port(2 + 2 * c, bufs[c]); p.port(3 + 2 * c, bufs[c])
            p.run(block)
            size = struct.unpack("<I", note[:4].tobytes())[0]
            outs.append(note[:8 + size].tobytes())
        rlen = t.ref(lambda: len(outs[1]))
        assert len(outs[0]) == rlen, (b, len(outs[0]), rlen)
        if t.live:
            assert outs[0] == outs[1], (b, next(i for i in range(len(outs[0])) if outs[0][i] != outs[1][i]))
        assert R.digest(outs[0]) == t.digest(lambda: outs[1]), b
        sizes.append(len(outs[0]))
    g.close(); r.close()
    return sizes


def test_descriptor_and_missing_urid_map():
    import meters_lv2_b200 as B
    mine, lib = descriptors(B.LIB_PATH)
    assert "EBUr128" in mine
    d = mine["EBUr128"]
    none = (C.POINTER(Feature) * 1)(None)
    assert not d.contents.instantiate(d, 48000.0, b"", none)               # no urid:map feature -> NULL (:140-144)


def test_silent_ui_no_messages(reftape):
    sizes = drive(reftape, {}, 6)
    assert set(sizes) == {16}                                               # bare sequence header while the UI is off


def test_gui_session_byte_parity(reftape):
    """UI connects, starts integration with dBTP on, changes radar time, pauses, resets, disconnects."""
    script = {
        1: [obj(MTR + b"meteron")],
        2: [cfg("UISETTINGS", 8 + 64), cfg("START", 0)],
        40: [cfg("RADARTIME", 30.0)],
        90: [cfg("PAUSE", 0)],
        95: [cfg("START", 0), cfg("RADARTIME", 10.0), cfg("RADARTIME", 700.0)],     # out-of-range: reply only
        140: [cfg("UISETTINGS", 8)],                                                   # dBTP off: tp_max -> -inf
        150: [cfg("RESET", 0)],
        170: [obj(MTR + b"meteroff")],
        175: [obj(MTR + b"meteron")],                                                  # resync of the stored radar, 16 points per cycle
    }
    sizes = drive(reftape, script, 210)
    assert max(sizes) > 1500 and sizes[0] == 16


def test_transport_follow_and_autoreset(reftape):
    script = {
        0: [obj(MTR + b"meteron"), cfg("TRANSPORTSYNC", 1.0), cfg("AUTORESET", 1.0)],
        5: [position(1.0)],
        30: [position(0.0)],
        33: [position(1.0)],                                                            # restart: auto reset -> RESETRADAR message
        50: [cfg("TRANSPORTSYNC", 0.0), position(0.0)],
        60: [cfg("AUTORESET", 0.0), cfg("START", 0)],
    }
    drive(reftape, script, 80)


def test_small_notify_buffer_and_odd_blocks(reftape):
    """capacity just above the reference's floor: histogram messages are rationed by the space left (:433)"""
    script = {0: [obj(MTR + b"meteron"), cfg("START", 0)]}
    drive(reftape, script, 120, block=1000, cap=1100)
    drive(reftape, script, 40, block=333, cap=4096, rate=44100.0)


def _levels(buf):
    """the 10 property values of the ebulevels object in a notify buffer -> {key urid: 4 value bytes}, or None"""
    size = struct.unpack("<I", buf[:4])[0]
    off, end, want = 16, 8 + size, urid(MTR + b"ebulevels")
    while off + 16 <= end:
        sz = struct.unpack("<I", buf[off + 8:off + 12])[0]
        oid, ot = struct.unpack("<II", buf[off + 16:off + 24])
        if ot == want:
            props, q = {}, off + 24
            while q + 16 <= off + 16 + sz:
                key, _ctx, vs, _vt = struct.unpack("<IIII", buf[q:q + 16])
                props[key] = bytes(buf[q + 16:q + 16 + vs])
                q += 16 + (vs + 7) // 8 * 8
            return props
        off += 16 + (sz + 7) // 8 * 8
    return None


def _level_bytes(buf, keys):
    """the 4-byte values of `keys` in the ebulevels object of a notify buffer, concatenated (empty if there is none)"""
    lv = _levels(buf)
    return np.frombuffer(b"".join(lv[k] for k in keys), np.uint8) if lv is not None else np.zeros(0, np.uint8)


def test_batched_mode_one_cycle_latency(monkeypatch, reftape):
    """B200M_LV2_BATCH: six EBUr128 instances share one bank; what each instance reports in cycle k + 1 is bit for bit what the
    reference plugin reports in cycle k (loudness values, ranges, true peak), with per-instance controls"""
    import meters_lv2_b200 as B
    monkeypatch.setenv("B200M_LV2_BATCH", "6")
    n, nb, blk = 6, 140, 1024
    mine, l1 = descriptors(B.LIB_PATH)
    ref, l2 = reftape.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    gs = [Plugin(mine["EBUr128"]) for _ in range(n)]
    rs = [reftape.obj(lambda: Plugin(ref["EBUr128"])) for _ in range(n)]
    x = S.white(2 * n, blk * nb, seed=61) * np.float32(3.0)
    x[2:4] *= np.float32(0.05)
    keys = [urid(MTR + k) for k in (b"ebu_loudnessM", b"ebu_maxloudnM", b"ebu_loudnessS", b"ebu_maxloudnS", b"ebu_integrated",
                                   b"ebu_range_min", b"ebu_range_max", b"truepeak", b"ebu_integrating")]
    script = {i: {} for i in range(n)}
    for i in range(n):
        script[i][1] = [obj(MTR + b"meteron")]
        script[i][2] = [cfg("UISETTINGS", 8 + 64 if i != 5 else 8), cfg("START", 0)]        # instance 5 never enables dBTP
    script[3][40] = [cfg("PAUSE", 0)]; script[3][55] = [cfg("START", 0)]
    script[4][70] = [cfg("RESET", 0)]
    empty = sequence([])
    notes_g = [np.zeros(CAP, np.uint8) for _ in range(n)]; notes_r = [np.zeros(CAP, np.uint8) for _ in range(n)]
    prev_ref = [None] * n
    checked = 0
    for b in range(nb):
        for plugs, notes in ((gs, notes_g), (rs, notes_r)):
            for i, p in enumerate(plugs):
                note = notes[i]
                note[:] = 0
                note[:8] = np.frombuffer(struct.pack("<II", CAP - 8, 0), np.uint8)
                ctl = sequence(script[i][b]) if b in script[i] else empty
                bufs = [np.ascontiguousarray(x[2 * i + c, b * blk:(b + 1) * blk]) for c in range(2)]
                p.port(0, ctl); p.port(1, note)
                for c in range(2):
                    p.port(2 + 2 * c, bufs[c]); p.port(3 + 2 * c, bufs[c])
                p.run(blk)
        for i in range(n):
            lg = _levels(notes_g[i].tobytes())
            lr = reftape.ref(lambda: _level_bytes(notes_r[i].tobytes(), keys[:8]))
            if lg is not None and prev_ref[i] is not None and b >= 4:
                for j, k in enumerate(keys[:8]):
                    v = prev_ref[i][4 * j:4 * j + 4].tobytes()
                    assert lg[k] == v, (b, i, k, struct.unpack("<f", lg[k]), struct.unpack("<f", v))
                checked += 1
            prev_ref[i] = lr if lr.size else None
    assert checked > n * 100
    for p in gs + rs:
        p.close()


@pytest.mark.timeout(180)
def test_batched_mode_survives_a_host_that_breaks_the_contract(monkeypatch):
    """a skipped instance, a changing block size and instances leaving in the middle must neither hang nor corrupt the others:
    a double submission (or a different n_samples) closes the open cycle as it is"""
    import meters_lv2_b200 as B
    monkeypatch.setenv("B200M_LV2_BATCH", "4")
    mine, l1 = descriptors(B.LIB_PATH)
    ps = [Plugin(mine["EBUr128"]) for _ in range(3)]                      # 3 members of a 4-slot hub
    x = S.white(6, 1024 * 60, seed=5)
    notes = [np.zeros(CAP, np.uint8) for _ in range(3)]
    on = sequence([obj(MTR + b"meteron"), cfg("START", 0)]); empty = sequence([])
    last = None
    for b in range(60):
        n = 512 if 30 <= b < 34 else 1024                                # the host changes its block size for a few cycles
        for i, p in enumerate(ps):
            if i == 1 and 10 <= b < 20:
                continue                                                 # instance 1 is bypassed for ten cycles
            if p is None:
                continue
            notes[i][:] = 0
            notes[i][:8] = np.frombuffer(struct.pack("<II", CAP - 8, 0), np.uint8)
            bufs = [np.ascontiguousarray(x[2 * i + c, b * 1024:b * 1024 + n]) for c in range(2)]
            p.port(0, on if b == 0 else empty); p.port(1, notes[i])
            for c in range(2):
                p.port(2 + 2 * c, bufs[c]); p.port(3 + 2 * c, bufs[c])
            p.run(n)
        if b == 45:
            ps[0].close(); ps[0] = None                                  # leaves while the others keep running
        lv = _levels(notes[2].tobytes())
        if lv is not None and b > 8:
            last = struct.unpack("<f", lv[urid(MTR + b"ebu_loudnessM")])[0]
            assert np.isfinite(last) and -40.0 < last < 10.0, (b, last)
    assert last is not None
    for p in ps:
        if p is not None:
            p.close()
    late = Plugin(mine["EBUr128"])                                       # a fresh hub can be created after the old one emptied
    late.close()
