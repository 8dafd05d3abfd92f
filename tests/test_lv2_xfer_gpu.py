"""GPU: the phasewheel / stereoscope LV2 plugins of libb200meters.so (csrc/lv2_xfer.cu) against the REFERENCE plugins
(src/xfer.c): byte-identical notify buffers (ui_state, rawstereo with both float vectors) and bit-identical phase port.
Without oracle/_ref the reference side is replayed from its recording (tests/_reftape.py): notify buffers by digest."""
import struct

import numpy as np
import pytest

import _oracle as O
import _reftape as R
import _signals as S
from test_lv2_ebur128_gpu import MTR, obj, sequence
from test_lv2_shim_gpu import descriptors, Plugin, u32

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,block,cap", [("phasewheel", 1024, 16384), ("stereoscope", 1024, 16384), ("phasewheel", 333, 8192), ("phasewheel", 1024, 8000)])
def test_xfer_plugins(name, block, cap, reftape):
    import meters_lv2_b200 as B
    t = reftape
    mine, l1 = descriptors(B.LIB_PATH)
    ref, l2 = t.obj(lambda: descriptors(O.PATHS["reference"]), 2)
    g, r = Plugin(mine[name]), t.obj(lambda: Plugin(ref[name]))
    nblocks = 30
    x = S.white(2, block * nblocks, seed=23); x[1] = 0.5 * x[0] + 0.5 * x[1]
    script = {3: [obj(MTR + b"ui_on")], 20: [obj(MTR + b"ui_off")], 25: [obj(MTR + b"ui_on")]}
    empty = sequence([])
    notes = [np.zeros(cap, np.uint8), np.zeros(cap, np.uint8)]
    phase = [np.zeros(1, np.float32), np.zeros(1, np.float32)]
    for b in range(nblocks):
        ctl = sequence(script[b]) if b in script else empty
        outs = []
        for p, note, ph in ((g, notes[0], phase[0]), (r, notes[1], phase[1])):
            note[:] = 0xA5
            note[:8] = np.frombuffer(struct.pack("<II", cap - 8, 0), np.uint8)
            bufs = [np.ascontiguousarray(x[c, b * block:(b + 1) * block]) for c in range(2)]
            p.port(0, ctl); p.port(1, note); p.port(6, ph)
            for c in range(2):
                p.port(2 + 2 * c, bufs[c]); p.port(3 + 2 * c, bufs[c])
            p.run(block)
            outs.append(note.tobytes())                        # whole buffer: a skipped cycle leaves it untouched on both sides
        size = t.ref(lambda: struct.unpack("<I", outs[1][:4])[0]).item()
        n = 8 + size if size <= cap - 8 and size != cap - 8 else cap
        if t.live:
            assert outs[0][:n] == outs[1][:n], b
        assert R.digest(outs[0][:n]) == t.digest(lambda: outs[1][:n]), b
        if name == "phasewheel":
            assert u32(phase[0])[0] == u32(t.ref(lambda: phase[1][0]))[0], b
    g.close(); r.close()
