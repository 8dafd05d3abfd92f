"""GPU: the bitmeter and SigDistHist LV2 plugins of libb200meters.so (csrc/lv2_stats.cu) against the REFERENCE plugins
(src/bitmeter.c, src/sigdistlv2.c compiled unmodified into oracle/_ref), driven like an LV2 host drives them; the
notify-port buffers (bim_stats with its 584-int vector, bim_information, sdh_histogram with its 361-int vector and
double mean / variance, sdh_information, control replies) must be identical bytes after every run()."""
import numpy as np
import pytest

import _signals as S
from test_lv2_ebur128_gpu import MTR, cfg, drive, obj, position

pytestmark = pytest.mark.gpu


def _audio(n, seed):
    x = S.white(2, n, seed=seed) * np.float32(1.7)
    x[0, 100:400] = 0.0                                     # zeros -> bim_zero
    x[0, 1000:1010] = np.float32(1e-41)                     # denormals
    x[0, 2000] = np.inf; x[0, 2001] = -np.inf; x[0, 2002] = np.nan
    x[0, 5000:9000] = np.round(x[0, 5000:9000] * 127) / np.float32(128)      # 8-bit material: few mantissa bits set
    return x


def test_bitmeter_windowed_average_reset(reftape):
    n, blk = 1024 * 120, 1024
    script = {
        2: [obj(MTR + b"meteron")],
        30: [cfg("AVERAGE", 0)],
        55: [cfg("PAUSE", 0)],
        60: [cfg("START", 0)],
        70: [cfg("RESET", 0)],
        85: [cfg("WINDOWED", 0)],
        100: [obj(MTR + b"meteroff")],
        110: [obj(MTR + b"meteron"), cfg("RESET", 0)],
    }
    sizes = drive(reftape, script, n // blk, block=blk, x=_audio(n, 5), cap=8192, name="bitmeter", nch=1)
    assert max(sizes) > 2400                                 # bim_stats carries the 584-int vector


def test_bitmeter_odd_blocks_44k1(reftape):
    drive(reftape, {0: [obj(MTR + b"meteron")]}, 90, block=441, x=_audio(441 * 90, 6), cap=4096, rate=44100.0, name="bitmeter", nch=1)


def test_sigdisthist_session(reftape):
    n, blk = 1024 * 100, 1024
    script = {
        1: [obj(MTR + b"meteron")],
        3: [cfg("START", 0)],
        40: [cfg("PAUSE", 0)],
        45: [cfg("UISETTINGS", 3.0), cfg("START", 0)],
        60: [cfg("RESET", 0)],
        70: [cfg("TRANSPORTSYNC", 1.0), cfg("AUTORESET", 1.0), position(0.0)],
        75: [position(1.0)],
        90: [position(0.0), obj(MTR + b"meteroff")],
    }
    x = S.white(2, n, seed=8) * np.float32(0.8)
    x[0, 3000:3100] = 5.0                                    # outside +-1.2: bins beyond the histogram are skipped
    sizes = drive(reftape, script, n // blk, block=blk, x=x, cap=8192, name="SigDistHist", nch=1)
    assert max(sizes) > 1500


def test_sigdisthist_small_blocks(reftape):
    drive(reftape, {0: [obj(MTR + b"meteron"), cfg("START", 0)]}, 200, block=64, x=S.white(2, 64 * 200, seed=9), cap=4096, name="SigDistHist", nch=1)
