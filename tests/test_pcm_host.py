"""CPU: the PCM ingest entry points (b200m_r128_run_*_pcm, b200m_pcm_convert) are exported, refuse bad arguments with
codes before touching a device, and without a device answer B200M_E_NODEVICE: there is no CPU conversion."""
import ctypes as C

import numpy as np
import pytest

E_INVAL, E_NODEVICE = -1, -5
PCM_NAMES = ("b200m_r128_run_device_pcm", "b200m_r128_run_host_pcm", "b200m_pcm_convert")
# a non-NULL pointer the library never dereferences: every call below fails its argument checks first
FAKE = C.c_void_p(0x1000)


def _lib():
    import meters_lv2_b200 as B
    return B, B.lib()


def test_pcm_symbols_exported():
    B, L = _lib()
    for n in PCM_NAMES:
        assert hasattr(L, n), n
        assert n in B.EXPORTS
    assert (B.PCM_F32, B.PCM_S16, B.PCM_S24, B.PCM_S32, B.PCM_PLANAR, B.PCM_INTERLEAVED) == (0, 1, 2, 3, 0, 16)


BAD_FMT = [4, 15, 5 | 16, 32, 1 | 32, 48, 0x100, 0xFFFFFFFF]


@pytest.mark.parametrize("fn", ["device", "host"])
def test_r128_pcm_argument_errors(fn):
    B, L = _lib()
    run = (lambda h, p, f, s, n: L.b200m_r128_run_device_pcm(h, p, f, s, n, None)) if fn == "device" else L.b200m_r128_run_host_pcm
    S16I = B.PCM_S16 | B.PCM_INTERLEAVED
    assert run(None, FAKE, S16I, 1024, 1024) == E_INVAL                    # NULL handle
    assert b"NULL" in L.b200m_last_error()
    assert run(FAKE, None, S16I, 1024, 1024) == E_INVAL                    # NULL input
    assert b"NULL" in L.b200m_last_error()
    for f in BAD_FMT:                                                      # bad type or layout code
        assert run(FAKE, FAKE, f, 1024, 1024) == E_INVAL, f
        assert b"format" in L.b200m_last_error()
    assert run(FAKE, FAKE, S16I, 1024, 0) == E_INVAL                       # nfram 0
    assert run(FAKE, FAKE, S16I, 8193, 8193) == E_INVAL                    # nfram 8193
    assert b"nfram" in L.b200m_last_error()
    assert run(FAKE, FAKE, S16I, 1023, 1024) == E_INVAL                    # stride < nfram
    assert b"stride" in L.b200m_last_error()
    # F32 | PLANAR is the float path itself: same checks
    assert run(None, FAKE, B.PCM_F32, 1024, 1024) == E_INVAL
    assert run(FAKE, FAKE, B.PCM_F32, 8, 9) == E_INVAL


def test_pcm_convert_argument_errors():
    B, L = _lib()
    cv = L.b200m_pcm_convert
    S24I = B.PCM_S24 | B.PCM_INTERLEAVED
    dst = C.c_void_p(0x2000)
    assert cv(0, None, S24I, 2, 4, 1024, 1024, dst, 1024, None) == E_INVAL          # NULL source
    assert cv(0, FAKE, S24I, 2, 4, 1024, 1024, None, 1024, None) == E_INVAL         # NULL destination
    for f in BAD_FMT:
        assert cv(0, FAKE, f, 2, 4, 1024, 1024, dst, 1024, None) == E_INVAL, f
    for nchan in (0, 9):
        assert cv(0, FAKE, S24I, nchan, 4, 1024, 1024, dst, 1024, None) == E_INVAL, nchan
    assert cv(0, FAKE, S24I, 2, 0, 1024, 1024, dst, 1024, None) == E_INVAL          # n_inst 0
    assert cv(0, FAKE, S24I, 2, 4, 1024, 0, dst, 1024, None) == E_INVAL             # nfram 0
    assert cv(0, FAKE, S24I, 2, 4, 8193, 8193, dst, 8196, None) == E_INVAL          # nfram 8193
    assert cv(0, FAKE, S24I, 2, 4, 1000, 1024, dst, 1024, None) == E_INVAL          # src_stride < nfram
    assert cv(0, FAKE, S24I, 2, 4, 1024, 1024, dst, 1020, None) == E_INVAL          # dst_stride < nfram
    assert cv(0, FAKE, S24I, 2, 4, 1024, 1024, dst, 1026, None) == E_INVAL          # rows not 16-byte aligned
    assert cv(0, FAKE, S24I, 2, 4, 1024, 1024, C.c_void_p(0x2004), 1024, None) == E_INVAL
    assert cv(0, C.c_void_p(0x1001), B.PCM_S16, 2, 4, 1024, 1024, dst, 1024, None) == E_INVAL   # int16 on an odd address
    assert cv(0, C.c_void_p(0x1002), B.PCM_S32, 2, 4, 1024, 1024, dst, 1024, None) == E_INVAL
    assert b"aligned" in L.b200m_last_error()


def test_pcm_convert_without_device_is_nodevice():
    import torch
    B, L = _lib()
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    # valid arguments (S24 may start on any byte): the only thing missing is the GPU
    rc = L.b200m_pcm_convert(0, C.c_void_p(0x1001), B.PCM_S24 | B.PCM_INTERLEAVED, 2, 4, 1024, 1024, C.c_void_p(0x2000), 1024, None)
    assert rc == E_NODEVICE
    assert b"no CUDA device" in L.b200m_last_error()


def test_python_layout_helper():
    """dtype -> format code, shapes and strides -> the ABI's stride convention (no device involved)"""
    B, _ = _lib()
    x = np.zeros((6, 100, 2), np.int16)
    p, fmt, stride, nfram, nseg, dev = B._pcm_layout(x[:, :96], True, 2)
    assert (fmt, stride, nfram, nseg, dev) == (B.PCM_S16 | B.PCM_INTERLEAVED, 100, 96, 6, False)
    y = np.zeros((4, 50, 3), np.uint8)
    assert B._pcm_layout(y[:, :7], False, 2)[1:5] == (B.PCM_S24, 50, 7, 4)
    z = np.zeros((3, 64, 2, 3), np.uint8)
    assert B._pcm_layout(z, True, 2)[1:5] == (B.PCM_S24 | B.PCM_INTERLEAVED, 64, 64, 3)
    assert B._pcm_layout(np.zeros((2, 8), np.int32), False, 2)[1:3] == (B.PCM_S32, 8)
    assert B._pcm_layout(np.zeros((2, 8), np.float32), False, 2)[1] == B.PCM_F32
    with pytest.raises(TypeError):
        B._pcm_layout(np.zeros((2, 8), np.float64), False, 2)
    with pytest.raises(ValueError):
        B._pcm_layout(np.zeros((2, 8, 2), np.int16)[:, :, :1], True, 1)      # channels not contiguous
    with pytest.raises(ValueError):
        B._pcm_layout(np.zeros((2, 8, 4), np.uint8), False, 2)               # 24-bit samples are 3 bytes
