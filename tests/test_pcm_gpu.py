"""GPU: PCM ingest.  b200m_pcm_convert hands the meters exactly the float32 numpy computes from the same PCM (bitwise, every
type x layout, odd channel counts and lengths, strided and minimally aligned sources), and an EBUr128 bank fed PCM through
run_pcm (host and device paths alternating) ends bit-identical to a bank fed numpy's float32 through the float path."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F32, S16, S24, S32 = 0, 1, 2, 3
PLANAR, INTERLEAVED = 0, 16
TYPES = {"f32": F32, "s16": S16, "s24": S24, "s32": S32}
ALIGN = {F32: 4, S16: 2, S24: 1, S32: 4}          # the smallest legal offset from a 256-byte aligned allocation
BITS = {S16: 16, S24: 24, S32: 32}

SPECIAL = {
    S16: [-32768, 32767, 0, -1, 1, -32767, 16384],
    S24: [-(1 << 23), (1 << 23) - 1, 0, -1, 1, -(1 << 23) + 1, 0x123456],
    # INT32 extremes, values that round to nearest even (2^24 + 1, odd values just below 2^31), their negatives
    S32: [-(1 << 31), (1 << 31) - 1, (1 << 24) + 1, (1 << 24) + 3, -(1 << 24) - 1, (1 << 31) - 65, (1 << 31) - 63,
          (1 << 31) - 129, (1 << 31) - 3, -(1 << 31) + 1, (1 << 25) + 2, (1 << 25) + 6, 0, -1],
    # NaN payloads (quiet, signalling, negative), -0, denormals, +-inf, largest finite
    F32: [0x7FC00001, 0x7F800001, 0xFFC12345, 0x7FFFFFFF, 0x80000000, 0x00000001, 0x807FFFFF, 0x00400000,
          0x7F800000, 0xFF800000, 0x7F7FFFFF, 0x00000000],
}


def u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def random_values(rng, t, shape, specials=True):
    """int32 sample values of type t (F32: their float32 bits as uint32), the type's special values first"""
    n = int(np.prod(shape))
    if t == F32:
        v = rng.uniform(-1.0, 1.0, n).astype(np.float32).view(np.uint32)
    else:
        lo, hi = -(1 << (BITS[t] - 1)), (1 << (BITS[t] - 1))
        v = rng.integers(lo, hi, n, dtype=np.int64)
    if specials:
        sp = np.array(SPECIAL[t], np.int64 if t != F32 else np.uint32)
        k = min(n, sp.size)
        v[:k] = sp[:k]
        v[-k:] = sp[:k][::-1]
    return v.reshape(shape)


def encode(v, t):
    """values -> the array a caller would hold: int16, int32, float32, or uint8 [..., 3] for packed 24-bit"""
    if t == S16:
        return v.astype(np.int16)
    if t == S32:
        return v.astype(np.int32)
    if t == F32:
        return np.asarray(v, np.uint32).view(np.float32)
    return np.ascontiguousarray(v.astype("<i4").view(np.uint8).reshape(*v.shape, 4)[..., :3])


def to_float(v, t):
    """numpy's conversion: what the header promises the meters see"""
    if t == F32:
        return np.asarray(v, np.uint32).view(np.float32)
    return v.astype(np.int32).astype(np.float32) * np.float32(2.0 ** -(BITS[t] - 1))


def planar_of(v_il):
    """[inst, nfram, nchan] -> [inst * nchan, nfram]"""
    n, f, c = v_il.shape
    return np.ascontiguousarray(v_il.transpose(0, 2, 1)).reshape(n * c, f)


# ---------------------------------------------------------------------------------------------------- conversion
@pytest.mark.parametrize("layout", ["planar", "interleaved"])
@pytest.mark.parametrize("tname", list(TYPES))
def test_pcm_convert_bitwise(tname, layout):
    import torch
    import meters_lv2_b200 as B
    t = TYPES[tname]
    il = layout == "interleaved"
    fmt = t | (INTERLEAVED if il else PLANAR)
    rng = np.random.default_rng(1000 + 10 * t + il)
    for nchan in (1, 2, 5, 8):
        for nfram in (1, 3, 1023, 8192):
            n_inst = 3
            stride = nfram + 5                                         # > nfram, and not a multiple of 4
            if il:
                v = random_values(rng, t, (n_inst, stride, nchan))
                want = planar_of(to_float(v[:, :nfram], t))
            else:
                v = random_values(rng, t, (n_inst * nchan, stride))
                want = to_float(v[:, :nfram], t)
            raw = encode(v, t).view(np.uint8).reshape(-1)
            off = ALIGN[t]
            buf = torch.zeros(raw.size + off + 64, dtype=torch.uint8, device="cuda")
            buf[off:off + raw.size] = torch.from_numpy(raw).cuda()
            dstride = ((nfram + 3) & ~3) + 4
            out = torch.full((n_inst * nchan, dstride), float("nan"), dtype=torch.float32, device="cuda")
            rc = B.lib().b200m_pcm_convert(0, C.c_void_p(buf.data_ptr() + off), fmt, nchan, n_inst, stride, nfram,
                                           C.c_void_p(out.data_ptr()), dstride, None)
            assert rc == 0, B.lib().b200m_last_error()
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            tag = (tname, layout, nchan, nfram)
            assert np.array_equal(u32(got[:, :nfram]), u32(want)), tag
            assert np.isnan(got[:, nfram:]).all(), tag                # nothing written past nfram
            # the Python mirror on a tensor view of the same bytes
            if t != S24:
                dt = {F32: torch.float32, S16: torch.int16, S32: torch.int32}[t]
                shape = (n_inst, stride, nchan) if il else (n_inst * nchan, stride)
                x = buf[off:off + raw.size].view(dt).view(shape)[:, :nfram]
                got2 = B.pcm_convert(x, il, nchan).cpu().numpy()
                assert np.array_equal(u32(got2), u32(want)), tag


def test_pcm_convert_s24_tensor_view():
    """uint8 [..., 3] tensors through pcm_convert, starting on an odd byte"""
    import torch
    import meters_lv2_b200 as B
    rng = np.random.default_rng(7)
    v = random_values(rng, S24, (4, 1030, 5))
    raw = encode(v, S24)                                               # [4, 1030, 5, 3]
    buf = torch.zeros(raw.size + 1, dtype=torch.uint8, device="cuda")
    buf[1:] = torch.from_numpy(raw.reshape(-1)).cuda()
    x = buf[1:].view(4, 1030, 5, 3)[:, :1027]
    got = B.pcm_convert(x, True, 5).cpu().numpy()
    assert np.array_equal(u32(got), u32(planar_of(to_float(v[:, :1027], S24))))


# ---------------------------------------------------------------------------------------------------- r128 parity
def pcm_block(rng, t, n_inst, nfram):
    """one block of an audio-like stereo stream: noise at a per-channel level, the type's extremes sprinkled in"""
    gain = 10.0 ** (-(3.0 + 40.0 * (np.arange(2 * n_inst) % 13) / 12.0) / 20.0)
    x = rng.uniform(-1.0, 1.0, (n_inst, nfram, 2)) * gain.reshape(n_inst, 1, 2)
    if t == F32:
        return x.astype(np.float32).view(np.uint32)
    full = float(1 << (BITS[t] - 1))
    v = np.clip(np.round(x * full), -full, full - 1).astype(np.int64)
    k = min(v.size, 4)
    v.reshape(-1)[:k] = [-(1 << (BITS[t] - 1)), (1 << (BITS[t] - 1)) - 1, -(1 << (BITS[t] - 1)), (1 << (BITS[t] - 1)) - 1][:k]
    return v


def layout_array(v_il, t, il, pad):
    """the caller's array for values [inst, nfram, 2], interleaved [inst, nfram + pad, 2] or planar [2 inst, nfram + pad];
    the block is [:, :nfram] of it (a strided view when pad > 0)"""
    n, nfram, _ = v_il.shape
    if il:
        full = np.zeros((n, nfram + pad, 2), v_il.dtype)
        full[:, :nfram] = v_il
    else:
        full = np.zeros((2 * n, nfram + pad), v_il.dtype)
        full[:, :nfram] = planar_of(v_il)
    return encode(full, t)


def float_rows_on_device(xf):
    """planar float32 on the device with the row layout of the bank's own conversion buffer (rows of a multiple of 64 floats):
    the tolerance-mode true-peak FIR picks its kernel by row alignment, so both banks must see the same one"""
    import torch
    nfram = xf.shape[1]
    d = torch.zeros((xf.shape[0], (nfram + 63) & ~63), dtype=torch.float32, device="cuda")
    d[:, :nfram] = torch.from_numpy(xf).cuda()
    return d[:, :nfram]


def snapshot_bytes(bank):
    """the bank's checkpoint blob written into a zeroed buffer: b200m_r128_snapshot leaves the padding that aligns each
    segment to 16 bytes unwritten, so blobs in uninitialised buffers differ there even between identical banks"""
    import meters_lv2_b200 as B
    n = B.lib().b200m_r128_snapshot_size(bank.h)
    buf = np.zeros(n, np.uint8)
    B._ck(B.lib().b200m_r128_snapshot(bank.h, B._np_ptr(buf), n, B._stream_ptr(None)))
    return buf


def state_equal(a, b, n_inst, all_hist):
    ra, ta = a.results()
    rb, tb = b.results()
    for k in ra.dtype.names:
        assert np.array_equal(ra[k].view(np.uint32), rb[k].view(np.uint32)), k
    assert np.array_equal(u32(ta), u32(tb)), "tp_max"
    for i in (range(n_inst) if all_hist else sorted({0, 1, n_inst // 2, n_inst - 1} | set(range(0, n_inst, 97)))):
        ha, hb = a.histogram(i), b.histogram(i)
        assert np.array_equal(ha[0], hb[0]) and np.array_equal(ha[1], hb[1]), "histograms of instance %d" % i
    assert np.array_equal(snapshot_bytes(a), snapshot_bytes(b)), "bank state"


BLOCKS = [1, 8192, 37, 1024, 4800, 3, 2048, 511, 8192, 1000, 4096, 777, 8192, 2400, 5, 8192, 640, 1024]
FORMATS = [(S16, True), (S24, True), (S32, True), (F32, True), (S16, False), (S24, False), (S32, False), (F32, False)]


@pytest.mark.parametrize("prec", ["exact", "fma"])
@pytest.mark.parametrize("n_inst", [1, 63, 64, 1000])
def test_r128_pcm_matches_float_path(n_inst, prec):
    import torch
    import meters_lv2_b200 as B
    mode = B.PREC_EXACT if prec == "exact" else B.PREC_FMA
    a, b = B.EBUr128(n_inst), B.EBUr128(n_inst)
    for g in (a, b):
        g.set_precision(mode)
        g.control(B.EBUr128.START)
    rng = np.random.default_rng(n_inst * 2 + mode)
    for j, nfram in enumerate(BLOCKS):
        t, il = FORMATS[j % len(FORMATS)]
        host = (j // len(FORMATS) + j) % 2 == 0                     # every format meets both paths
        pad = 0 if j % 3 else 3                                      # every third block from a strided array
        v = pcm_block(rng, t, n_inst, nfram)
        xf = np.ascontiguousarray(planar_of(to_float(v, t)))
        xp = layout_array(v, t, il, pad)
        if host:
            a.run(xf)
            b.run_pcm(xp[:, :nfram], il)
        else:
            a.run(float_rows_on_device(xf))
            b.run_pcm(torch.from_numpy(xp).cuda()[:, :nfram], il)
    torch.cuda.synchronize()
    state_equal(a, b, n_inst, all_hist=True)


def test_r128_pcm_full_size():
    """8192 stereo instances: S16 interleaved through run_host_pcm (pinned buffers), S24 interleaved through run_device_pcm,
    48 blocks of 1024 frames each, every result bit-identical to the float path fed numpy's conversion"""
    import torch
    import meters_lv2_b200 as B
    n, nfram, nb = 8192, 1024, 48
    banks = {k: B.EBUr128(n) for k in ("a16", "b16", "a24", "b24")}
    for g in banks.values():
        g.set_precision(B.PREC_FMA)
        g.control(B.EBUr128.START)
    rng = np.random.default_rng(8192)
    pinned = [B.host_alloc(n, nfram) for _ in range(2)]            # float32 [n, nfram] = n x nfram x 2 int16
    for s in range(nb):
        v16 = pcm_block(rng, S16, n, nfram)
        hb = pinned[s % 2].view(np.int16).reshape(n, nfram, 2)
        torch.cuda.synchronize()                                     # the previous use of this buffer has been copied
        hb[:] = v16
        banks["a16"].run(np.ascontiguousarray(planar_of(to_float(v16, S16))))
        banks["b16"].run_pcm(hb, True)
        v24 = pcm_block(rng, S24, n, nfram)
        banks["a24"].run(float_rows_on_device(planar_of(to_float(v24, S24))))
        banks["b24"].run_pcm(torch.from_numpy(encode(v24, S24)).cuda(), True)
    torch.cuda.synchronize()
    state_equal(banks["a16"], banks["b16"], n, all_hist=False)
    state_equal(banks["a24"], banks["b24"], n, all_hist=False)
    r, _ = banks["b16"].results()
    assert np.isfinite(r["integrated"]).all() and (r["hist_M_count"] > 0).all()
