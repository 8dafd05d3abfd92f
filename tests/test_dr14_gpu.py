"""GPU: DR-14 / TPnRMS (csrc/dr14.cu, csrc/lv2_dr14.cu) against the REFERENCE plugins dr14stereo / dr14mono /
TPnRMSstereo (src/dr14.c compiled unmodified into oracle/_ref), driven through their own LV2 run().  Every output port
(dB values, DR scores, block count) must be bit-identical after every cycle; in cycles where the reference writes a
rand()-based block count (GUI re-init) only the regime is compared.  Without oracle/_ref the reference side is replayed from
its recording (tests/_reftape.py)."""
import struct

import numpy as np
import pytest

import _oracle as O
import _signals as S
from test_lv2_ebur128_gpu import ATOM, MTR, obj, position, sequence
from test_lv2_shim_gpu import descriptors, Plugin, u32

pytestmark = pytest.mark.gpu
OUT_ST = [3, 6, 7, 8, 9, 10, 13, 14, 15, 16, 17, 18]          # DRPortIndex outputs (src/dr14.c:27-43)
OUT_MONO = [3, 6, 7, 8, 9, 10]


def _music(nch, n, seed, gain):
    """noise with a slow loudness envelope so that the 3 s windows differ (exercises the top-20 % selection)"""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 48000.0
    env = (0.25 + 0.75 * np.abs(np.sin(2 * np.pi * t / 7.3 + seed))).astype(np.float32)
    return (rng.uniform(-1, 1, (nch, n)).astype(np.float32) * env * np.float32(gain)).astype(np.float32)


def _connect(p, nch, ctl, ctrl, bufs, outs):
    p.port(0, ctl); p.port(1, ctrl[0]); p.port(2, ctrl[1])
    for i, a in outs.items():
        p.port(i, a)
    p.port(4, bufs[0]); p.port(5, bufs[0])
    if nch == 2:
        p.port(11, bufs[1]); p.port(12, bufs[1])


def _side_by_side(t, name, nch, nblocks, block, script=None, x=None, rate=48000.0):
    import meters_lv2_b200 as B
    mine, l1 = descriptors(B.LIB_PATH)
    ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    g, r = Plugin(mine[name], rate), t.obj(lambda: Plugin(ref[name], rate))
    ports = OUT_ST if nch == 2 else OUT_MONO
    if x is None:
        x = _music(nch, nblocks * block, 3, 0.7)
    script = script or {}
    empty = sequence([])
    go = {i: np.zeros(1, np.float32) for i in ports}; ro = {i: np.zeros(1, np.float32) for i in ports}
    gc = [np.ones(1, np.float32), np.zeros(1, np.float32)]; rc = [np.ones(1, np.float32), np.zeros(1, np.float32)]
    for b in range(nblocks):
        ev = script.get(b, {})
        ctl = sequence(ev.get("atoms", [])) if ev.get("atoms") else empty
        for c in (gc, rc):
            c[0][0] = ev.get("follow", c[0][0]); c[1][0] = ev.get("reset", 0.0)
        for p, c, o in ((g, gc, go), (r, rc, ro)):
            bufs = [np.ascontiguousarray(x[k, b * block:(b + 1) * block]) for k in range(nch)]
            _connect(p, nch, ctl, c, bufs, o)
            p.run(block)
        rv = dict(zip(ports, t.ref(lambda: [ro[i][0] for i in ports])))
        for i in ports:
            if i == 3 and rv[i] < 0:                        # -1 - (rand () & 0xffff): same regime only
                assert go[i][0] < 0, (name, b)
            else:
                assert u32(go[i])[0] == u32(rv[i])[0], (name, b, i, go[i][0], rv[i])
    g.close(); r.close()
    return rv


def test_dr14_stereo_plugin_45s(reftape):
    ro = _side_by_side(reftape, "dr14stereo", 2, 270, 8192)   # 46 s: 15 windows, DR valid after 3
    assert 1.0 <= ro[18] <= 20.0 and ro[3] == 45.0


def test_dr14_mono_odd_blocks_and_44k1(reftape):
    _side_by_side(reftape, "dr14mono", 1, 700, 1000, rate=44100.0)


def test_dr14_controls_transport_reset_gui(reftape):
    script = {
        20: dict(atoms=[position(1.0)]),                        # transport starts, follow = 1 -> reset_peaks
        60: dict(atoms=[obj(MTR + b"meteron")]),                # GUI re-init values every cycle until meteroff
        64: dict(atoms=[obj(MTR + b"meteroff")]),
        90: dict(reset=1.0),                                    # reset button
        120: dict(atoms=[obj(MTR + b"dr14reset")]),
        150: dict(follow=0.0, atoms=[position(0.0)]),
        155: dict(atoms=[position(1.0)]),                       # follow off: no reset
    }
    _side_by_side(reftape, "dr14stereo", 2, 200, 4096, script)


def test_dr14_silence_nan_and_loud(reftape):
    n, blk = 8192 * 60, 8192
    x = _music(2, n, 5, 0.9)
    x[:, 8192 * 10:8192 * 30] = 0.0                              # 3 s windows of silence: not scored, peak_cur kept
    x[0, 8192 * 40 + 5] = np.nan                                 # NaN poisons one window's rms_sum
    x[1, 8192 * 50:8192 * 52] *= np.float32(3.0)                 # > 0 dBFS: histogram clamps at the top bin
    _side_by_side(reftape, "dr14stereo", 2, 60, blk, x=x)


def test_tpnrms_plugins(reftape):
    _side_by_side(reftape, "TPnRMSstereo", 2, 40, 1024, {10: dict(reset=1.0), 20: dict(atoms=[obj(MTR + b"meteron")]), 22: dict(atoms=[obj(MTR + b"meteroff")])})
    _side_by_side(reftape, "TPnRMSmono", 1, 30, 777)


@pytest.mark.parametrize("wide", [False, True, "slabs"])
def test_dr14_bank_vs_reference_instances(wide, monkeypatch, reftape):
    """the batch API: 5 stereo instances in one bank vs 5 reference plugin instances; `wide` forces the 64-channel CTA form of the
    process() kernel (csrc/tpk.cu: every warp carries ballistics / K-meter / DR lanes) that large banks get by default"""
    import torch
    import meters_lv2_b200 as B
    if wide == "slabs":
        monkeypatch.setenv("B200M_TPK_SLAB", "192"); monkeypatch.setenv("B200M_TPK_SPLIT", "2")   # 8192-frame blocks in 43 slabs: DR window ends fall inside slabs
    elif wide:
        monkeypatch.setenv("B200M_TPK_WIDE", "2"); monkeypatch.setenv("B200M_TPK_SPLIT", "0")
    t = reftape
    ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    ninst, nblocks, blk = 5, 150, 8192
    gains = [0.9, 0.3, 0.05, 1e-5, 0.6]                          # instance 3 stays below the silence gate
    x = np.concatenate([_music(2, nblocks * blk, 10 + i, gains[i]) for i in range(ninst)], axis=0)
    bank = B.DR14(ninst, 2, 48000.0, True)
    xd = torch.from_numpy(x).cuda()
    plugs = [t.obj(lambda: Plugin(ref["dr14stereo"], 48000.0)) for _ in range(ninst)]
    empty = sequence([])
    outs = [{i: np.zeros(1, np.float32) for i in OUT_ST} for _ in range(ninst)]
    ctrl = [np.ones(1, np.float32), np.zeros(1, np.float32)]
    last = [None] * ninst
    for b in range(nblocks):
        bank.run(xd[:, b * blk:(b + 1) * blk])
        res = bank.results()
        for i, p in enumerate(plugs):
            bufs = [np.ascontiguousarray(x[2 * i + k, b * blk:(b + 1) * blk]) for k in range(2)]
            _connect(p, 2, empty, ctrl, bufs, outs[i])
            p.run(blk)
            o = last[i] = dict(zip(OUT_ST, t.ref(lambda: [outs[i][k] for k in OUT_ST])))
            want = dict(v_peak=(o[6][0], o[13][0]), m_peak=(o[7][0], o[14][0]), v_rms=(o[8][0], o[15][0]), m_rms=(o[9][0], o[16][0]), dr=(o[10][0], o[17][0]))
            for k, (a0, a1) in want.items():
                assert u32(res[k][i])[0] == u32(np.float32(a0))[()] and u32(res[k][i])[1] == u32(np.float32(a1))[()], (b, i, k, res[k][i], a0, a1)
            assert u32(res["dr_total"][i:i + 1])[0] == u32(o[18])[0] and u32(res["block_count"][i:i + 1])[0] == u32(o[3])[0], (b, i)
    h = bank.histogram(0, 0)
    o0, o3 = last[0], last[3]
    assert h.sum() == int(o0[3][0] / 3)                          # one histogram entry per scored window
    assert o3[3][0] == 0.0                                       # the silent instance never scored
    for p in plugs:
        p.close()
