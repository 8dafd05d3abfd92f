"""meters.lv2_b200 — host-side mirror (Python/ctypes) of the b200meters C ABI (include/b200meters.h).

The product is the CUDA library `libb200meters.so` built in-tree from csrc/ by build.py; this module
only binds its C entry points for tests and bench.py.  Class and method names follow the reference's
DSP classes (Ebu_r128_proc, TruePeakdsp, Kmeterdsp, Stcorrdsp, the spectr30 plugin, the phasewheel
FFT analysis), each batched over N instances.  There is no CPU path: constructing a bank without the
built library or without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200meters.so")
HIST_LEN = 751
MIX_WORDS = 1508
MAX_BLOCK = 8192
_v = C.c_void_p
_lib = None


class B200MError(RuntimeError):
    pass


class EbuResult(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("loudness_M", "maxloudn_M", "loudness_S", "maxloudn_S", "integrated",
                                          "integ_thr", "range_min", "range_max", "range_thr")] + \
               [("hist_M_count", C.c_int32), ("hist_S_count", C.c_int32), ("frag_power", C.c_float)]


EBU_RESULT_DTYPE = np.dtype([(n, "<f4") for n in ("loudness_M", "maxloudn_M", "loudness_S", "maxloudn_S", "integrated",
                                                    "integ_thr", "range_min", "range_max", "range_thr")] +
                            [("hist_M_count", "<i4"), ("hist_S_count", "<i4"), ("frag_power", "<f4")])
TPK_RESULT_DTYPE = np.dtype([("tp_m", "<f4"), ("tp_p", "<f4"), ("km_rms", "<f4"), ("km_peak", "<f4")])

_PROTOS = {
    "b200m_abi_version": (C.c_int, []),
    "b200m_last_error": (C.c_char_p, []),
    "b200m_device_count": (C.c_int, []),
    "b200m_host_alloc": (C.c_int, [C.POINTER(_v), C.c_size_t]),
    "b200m_host_free": (C.c_int, [_v]),
    "b200m_launch_count": (C.c_uint64, []),
    "b200m_peak_probe": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "b200m_design_ebu": (C.c_int, [C.c_float, _v]),
    "b200m_design_tpk": (C.c_int, [C.c_float, _v, _v, _v]),
    "b200m_design_cor": (C.c_int, [C.c_int, C.c_float, C.c_float, _v]),
    "b200m_design_spec": (C.c_int, [C.c_double, _v]),
    # EBU
    "b200m_ebu_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_uint32, C.c_float]),
    "b200m_ebu_destroy": (C.c_int, [_v]),
    "b200m_ebu_reset": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_ebu_integr_start": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_ebu_integr_pause": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_ebu_integr_reset": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_ebu_process_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_ebu_process_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_ebu_results": (C.c_int, [_v, _v, _v]),
    "b200m_ebu_histogram": (C.c_int, [_v, C.c_uint32, _v, _v, _v]),
    "b200m_ebu_coeffs": (C.c_int, [_v, _v]),
    "b200m_ebu_state": (C.c_int, [_v, C.c_uint32, _v, _v, _v, _v, _v]),
    "b200m_ebu_mix_reduce": (C.c_int, [_v, _v, _v]),
    "b200m_ebu_mix_finish": (C.c_int, [_v, _v, _v, _v]),
    # True peak + K-meter
    "b200m_tpk_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_float, C.c_uint32]),
    "b200m_tpk_destroy": (C.c_int, [_v]),
    "b200m_tpk_process_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, C.c_uint32, _v]),
    "b200m_tpk_process_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, C.c_uint32]),
    "b200m_tpk_read_device": (C.c_int, [_v, _v]),
    "b200m_selftest_log10f": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32, _v, _v]),
    "b200m_lv2_gon_layout": (C.c_int, [_v, C.c_int]),
    "b200m_ebu_clear": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_tpk_clear": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_spec_set_precision": (C.c_int, [_v, C.c_int]),
    "b200m_cor_set_precision": (C.c_int, [_v, C.c_int]),
    "b200m_pw_debug_capture": (C.c_int, [_v, C.c_int]),
    "b200m_pw_attach_cor": (C.c_int, [_v, _v]),
    "b200m_tpk_set_precision": (C.c_int, [_v, C.c_int]),
    "b200m_tpk_precision": (C.c_int, [_v]),
    "b200m_tpk_results": (C.c_int, [_v, _v, _v]),
    "b200m_tpk_reset": (C.c_int, [_v, C.c_int32, _v]),
    "b200m_tpk_reset_kmeter": (C.c_int, [_v, _v]),
    "b200m_tpk_coeffs": (C.c_int, [_v, _v, _v, _v]),
    "b200m_tpk_state": (C.c_int, [_v, _v, _v, _v, _v, _v, _v, _v]),
    "b200m_tpk_debug_capture": (C.c_int, [_v, C.c_int]),
    "b200m_tpk_debug_timeline": (C.c_int, [_v, _v, C.c_int]),
    "b200m_tpk_debug_upsampled": (C.c_int, [_v, C.c_uint32, _v, C.c_uint32, _v]),
    # EBUr128 plugin cycle
    "b200m_r128_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_float, C.c_int]),
    "b200m_r128_destroy": (C.c_int, [_v]),
    "b200m_r128_control": (C.c_int, [_v, C.c_int32, C.c_int, _v]),
    "b200m_r128_run_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_r128_run_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_r128_run_device_pcm": (C.c_int, [_v, _v, C.c_uint32, C.c_size_t, C.c_uint32, _v]),
    "b200m_r128_run_host_pcm": (C.c_int, [_v, _v, C.c_uint32, C.c_size_t, C.c_uint32]),
    "b200m_pcm_convert": (C.c_int, [C.c_int, _v, C.c_uint32, C.c_uint32, C.c_uint32, C.c_size_t, C.c_uint32, _v, C.c_size_t, _v]),
    "b200m_r128_results": (C.c_int, [_v, _v, _v, _v]),
    "b200m_r128_set_dbtp": (C.c_int, [_v, C.c_int]),
    "b200m_r128_set_precision": (C.c_int, [_v, C.c_int]),
    "b200m_r128_histogram": (C.c_int, [_v, C.c_uint32, _v, _v, _v]),
    "b200m_r128_snapshot_size": (C.c_size_t, [_v]),
    "b200m_r128_snapshot": (C.c_int, [_v, _v, C.c_size_t, _v]),
    "b200m_r128_restore": (C.c_int, [_v, _v, C.c_size_t, _v]),
    "b200m_ebu_snapshot_size": (C.c_size_t, [_v]),
    "b200m_ebu_snapshot": (C.c_int, [_v, _v, C.c_size_t, _v]),
    "b200m_ebu_restore": (C.c_int, [_v, _v, C.c_size_t, _v]),
    "b200m_tpk_snapshot_size": (C.c_size_t, [_v]),
    "b200m_tpk_snapshot": (C.c_int, [_v, _v, C.c_size_t, _v]),
    "b200m_tpk_restore": (C.c_int, [_v, _v, C.c_size_t, _v]),
    "b200m_r128_ebu": (_v, [_v]),
    "b200m_r128_tpk": (_v, [_v]),
    # Stcorr
    "b200m_dr14_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_uint32, C.c_double, C.c_int]),
    "b200m_dr14_destroy": (C.c_int, [_v]),
    "b200m_dr14_run_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_dr14_run_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_dr14_reset": (C.c_int, [_v, _v]),
    "b200m_dr14_results": (C.c_int, [_v, _v, _v]),
    "b200m_dr14_histogram": (C.c_int, [_v, C.c_uint32, C.c_uint32, _v, _v]),
    "b200m_cor_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_int, C.c_float, C.c_float]),
    "b200m_cor_destroy": (C.c_int, [_v]),
    "b200m_cor_process_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_cor_process_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_cor_results": (C.c_int, [_v, _v, _v]),
    "b200m_cor_state": (C.c_int, [_v, _v, _v]),
    "b200m_cor_coeffs": (C.c_int, [_v, _v]),
    # needle-meter ballistics
    "b200m_ppm_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_float, C.c_int]),
    "b200m_ppm_destroy": (C.c_int, [_v]),
    "b200m_ppm_set_gain": (C.c_int, [_v, C.c_float, C.c_float]),
    "b200m_ppm_process_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_ppm_process_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_ppm_read_device": (C.c_int, [_v, _v]),
    "b200m_ppm_results": (C.c_int, [_v, _v, _v]),
    "b200m_ppm_state": (C.c_int, [_v, _v, _v]),
    "b200m_design_ppm": (C.c_int, [C.c_int, C.c_float, _v]),
    # bit-meter, signal distribution histogram
    "b200m_bim_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_double]),
    "b200m_bim_destroy": (C.c_int, [_v]),
    "b200m_bim_control": (C.c_int, [_v, C.c_int, _v]),
    "b200m_bim_run_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_bim_run_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_bim_results": (C.c_int, [_v, C.c_uint32, _v, _v, _v, _v, _v]),
    "b200m_bim_window_closed": (C.c_int, [_v]),
    "b200m_bim_published": (C.c_int, [_v, C.c_uint32, _v, _v, _v, _v, _v]),
    "b200m_sdh_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_double]),
    "b200m_sdh_destroy": (C.c_int, [_v]),
    "b200m_sdh_control": (C.c_int, [_v, C.c_int, _v]),
    "b200m_sdh_run_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, _v]),
    "b200m_sdh_run_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32]),
    "b200m_sdh_results": (C.c_int, [_v, C.c_uint32, _v, _v, _v, _v, _v]),
    # spectr30
    "b200m_spec_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_uint32, C.c_double]),
    "b200m_spec_destroy": (C.c_int, [_v]),
    "b200m_spec_process_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, C.c_float, C.c_float, _v]),
    "b200m_spec_process_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, C.c_float, C.c_float]),
    "b200m_spec_results": (C.c_int, [_v, _v, _v]),
    "b200m_spec_state": (C.c_int, [_v, C.c_uint32, _v, _v, _v, _v]),
    "b200m_spec_coeffs": (C.c_int, [_v, _v]),
    # phasewheel
    "b200m_pw_create": (C.c_int, [C.POINTER(_v), C.c_int, C.c_uint32, C.c_uint32, C.c_double]),
    "b200m_pw_set_mode": (C.c_int, [_v, C.c_int]),
    "b200m_pw_destroy": (C.c_int, [_v]),
    "b200m_pw_process_device": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, C.c_float, C.POINTER(C.c_int), _v]),
    "b200m_pw_process_host": (C.c_int, [_v, _v, C.c_size_t, C.c_uint32, C.c_float, C.POINTER(C.c_int)]),
    "b200m_pw_results": (C.c_int, [_v, _v, _v, _v, _v]),
    "b200m_pw_raw": (C.c_int, [_v, C.c_uint32, _v, _v, _v, _v, _v]),
    "b200m_pw_device_results": (C.c_int, [_v, C.POINTER(_v), C.POINTER(_v), C.POINTER(_v)]),
}
EXPORTS = tuple(_PROTOS)


def lib():
    """Load libb200meters.so (fails loudly if it has not been built: there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200MError("%s is missing: run `python meters.lv2_b200/build.py` "
                             "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            try:
                fn = getattr(L, name)
            except AttributeError:      # reported by missing_exports(); calling it raises AttributeError
                continue
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def missing_exports():
    """Names declared in include/b200meters.h that the built library does not export."""
    L = lib()
    return [n for n in _PROTOS if not hasattr(L, n)]


def _ck(rc):
    if rc != 0:
        raise B200MError("b200meters error %d: %s" % (rc, lib().b200m_last_error().decode()))


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _dev_ptr(x):
    """torch CUDA tensor | int device pointer -> (pointer, row stride in floats, rows, cols)."""
    if isinstance(x, int):
        raise TypeError("pass (ptr, stride, nfram) explicitly via process_ptr()")
    assert x.is_cuda and x.dim() == 2 and x.stride(1) == 1, "need a [channels, nfram] float32 CUDA tensor"
    stride = x.stride(0) if x.shape[0] > 1 else max(x.stride(0), x.shape[1])   # 1-row tensors may report stride 0/1
    return C.c_void_p(x.data_ptr()), stride, x.shape[0], x.shape[1]


def _stream_ptr(stream):
    if stream is None:
        try:
            import torch
            if torch.cuda.is_available():
                return C.c_void_p(torch.cuda.current_stream().cuda_stream)
        except ImportError:
            pass
        return C.c_void_p(0)
    if isinstance(stream, int):
        return C.c_void_p(stream)
    return C.c_void_p(stream.cuda_stream)


def _host_planar(x):
    """numpy [channels, nfram] float32 (row-contiguous) or a pinned torch CPU tensor."""
    if isinstance(x, np.ndarray):
        assert x.dtype == np.float32 and x.ndim == 2 and x.strides[1] == 4
        stride = x.strides[0] // 4 if x.shape[0] > 1 else max(x.strides[0] // 4, x.shape[1])
        return _np_ptr(x), stride, x.shape[0], x.shape[1]
    assert (not x.is_cuda) and x.dim() == 2 and x.stride(1) == 1
    return C.c_void_p(x.data_ptr()), x.stride(0), x.shape[0], x.shape[1]


PCM_F32, PCM_S16, PCM_S24, PCM_S32 = 0, 1, 2, 3
PCM_PLANAR, PCM_INTERLEAVED = 0, 16
_PCM_BYTES = {PCM_F32: 4, PCM_S16: 2, PCM_S24: 3, PCM_S32: 4}


def _pcm_layout(x, interleaved, nchan):
    """numpy array or torch tensor of PCM -> (pointer, fmt, stride, nfram, segments, on_device).

    The dtype selects the sample type: float32, int16, int32, or uint8 with a last dimension of 3 (packed little-endian
    24-bit).  Planar: [rows, nfram] (rows = instances x nchan); interleaved: [instances, nfram, nchan].  Only the outer
    dimension may be strided; `stride` comes back in elements (planar) or frames (interleaved), as the C ABI counts it."""
    if isinstance(x, np.ndarray):
        name, shape, bstrides, ptr, dev = x.dtype.name, x.shape, x.strides, x.ctypes.data, False
    else:
        name = str(x.dtype).replace("torch.", "")
        shape, bstrides, ptr, dev = tuple(x.shape), tuple(s * x.element_size() for s in x.stride()), x.data_ptr(), x.is_cuda
    types = {"float32": PCM_F32, "int16": PCM_S16, "int32": PCM_S32, "uint8": PCM_S24}
    if name not in types:
        raise TypeError("PCM dtype must be float32, int16, int32 or uint8 (packed 24-bit), not %s" % name)
    t = types[name]
    bps = _PCM_BYTES[t]
    if t == PCM_S24:
        if shape[-1] != 3 or bstrides[-1] != 1:
            raise ValueError("24-bit PCM is a uint8 array whose last dimension holds the 3 bytes of a sample")
        shape, bstrides = shape[:-1], bstrides[:-1]
    inner = (nchan,) if interleaved else ()
    if len(shape) != 2 + len(inner) or tuple(shape[2:]) != inner:
        raise ValueError("PCM shape %s: want %s" % (shape, "[instances, nfram, %d]" % nchan if interleaved else "[rows, nfram]"))
    frame_bytes = bps * (nchan if interleaved else 1)
    if bstrides[1] != frame_bytes or (interleaved and bstrides[2] != bps):
        raise ValueError("PCM frames and channels must be contiguous (only the outer dimension may be strided)")
    nseg, nfram = shape[0], shape[1]
    stride = bstrides[0] // frame_bytes if nseg > 1 else nfram
    if nseg > 1 and bstrides[0] % frame_bytes:
        raise ValueError("PCM row pitch is not a whole number of frames")
    return ptr, t | (PCM_INTERLEAVED if interleaved else PCM_PLANAR), stride, nfram, nseg, dev


def pcm_convert(x, interleaved, nchan=2, out=None, stream=None):
    """b200m_pcm_convert: a CUDA tensor of PCM (layouts of _pcm_layout) -> planar float32 rows [instances x nchan, nfram]
    on the same device, the values every bank is fed (the header's conversion table).  `out` may be a row-strided view
    (16-byte aligned, row stride a multiple of 4)."""
    import torch
    p, fmt, stride, nfram, nseg, dev = _pcm_layout(x, interleaved, nchan)
    if not dev:
        raise ValueError("pcm_convert takes CUDA tensors; EBUr128.run_pcm takes host arrays")
    n_inst = nseg if interleaved else nseg // nchan
    if not interleaved and nseg % nchan:
        raise ValueError("%d planar rows are not whole instances of %d channels" % (nseg, nchan))
    if out is None:
        out = torch.empty((n_inst * nchan, (nfram + 3) & ~3), dtype=torch.float32, device=x.device)[:, :nfram]
    o, ostride, rows, n = _dev_ptr(out)
    assert out.dtype == torch.float32 and rows == n_inst * nchan and n == nfram
    _ck(lib().b200m_pcm_convert(x.device.index or 0, C.c_void_p(p), fmt, nchan, n_inst, stride, nfram, o, ostride, _stream_ptr(stream)))
    return out


def design_ebu(fsamp):
    o = np.empty(7, np.float32)
    _ck(lib().b200m_design_ebu(fsamp, _np_ptr(o)))
    return o


def design_tpk(fsamp):
    w = np.empty(4, np.float32); t = np.empty(120, np.float32); k = np.empty(2, np.float32)
    _ck(lib().b200m_design_tpk(fsamp, _np_ptr(w), _np_ptr(t), _np_ptr(k)))
    return w, t, k


def design_cor(fsamp, flp=2e3, tcf=0.3):
    w = np.empty(2, np.float32)
    _ck(lib().b200m_design_cor(int(fsamp), flp, tcf, _np_ptr(w)))
    return w


def design_spec(rate):
    W = np.empty((30, 6, 6), np.float64)
    _ck(lib().b200m_design_spec(rate, _np_ptr(W)))
    return W


def host_alloc(rows, cols):
    """[rows, cols] float32 numpy array in pinned host memory from b200m_host_alloc (placed on the GPU-local NUMA node);
    freed with b200m_host_free when the array is garbage-collected."""
    import weakref
    p = _v()
    nbytes = int(rows) * int(cols) * 4
    _ck(lib().b200m_host_alloc(C.byref(p), nbytes))
    buf = (C.c_float * (int(rows) * int(cols))).from_address(p.value)
    a = np.frombuffer(buf, dtype=np.float32).reshape(int(rows), int(cols))
    weakref.finalize(buf, lib().b200m_host_free, _v(p.value))
    return a


def peak_probe(kind, device=0):
    """kind 0: fp32 unfused mul+add, kind 1: fp64; returns 1e9 lane-ops/s measured on the device."""
    v = C.c_double(0)
    _ck(lib().b200m_peak_probe(device, kind, C.byref(v)))
    return v.value


def launch_count():
    return int(lib().b200m_launch_count())


class _Bank:
    _destroy = None

    def __init__(self):
        self.h = _v()

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            if self._destroy:
                getattr(lib(), self._destroy)(self.h)
            self.h = _v()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Ebu_r128_proc(_Bank):
    """N x LV2M::Ebu_r128_proc (ebumeter/ebu_r128_proc.h:66-125)."""
    _destroy = "b200m_ebu_destroy"

    def __init__(self, n_inst, nchan=2, fsamp=48000.0, device=0):
        super().__init__()
        self.n_inst, self.nchan = n_inst, nchan
        _ck(lib().b200m_ebu_create(C.byref(self.h), device, n_inst, nchan, fsamp))

    def reset(self, stream=None):
        _ck(lib().b200m_ebu_reset(self.h, -1, _stream_ptr(stream)))

    def integr_start(self, inst=-1, stream=None):
        _ck(lib().b200m_ebu_integr_start(self.h, inst, _stream_ptr(stream)))

    def integr_pause(self, inst=-1, stream=None):
        _ck(lib().b200m_ebu_integr_pause(self.h, inst, _stream_ptr(stream)))

    def integr_reset(self, inst=-1, stream=None):
        _ck(lib().b200m_ebu_integr_reset(self.h, inst, _stream_ptr(stream)))

    def process(self, x, stream=None):
        """x: [n_inst*nchan, nfram] float32 CUDA tensor (device path) or numpy/pinned CPU (host path)."""
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == self.n_inst * self.nchan
            _ck(lib().b200m_ebu_process_host(self.h, p, s, n))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == self.n_inst * self.nchan
            _ck(lib().b200m_ebu_process_device(self.h, p, s, n, _stream_ptr(stream)))

    def process_ptr(self, ptr, stride, nfram, stream=None):
        _ck(lib().b200m_ebu_process_device(self.h, C.c_void_p(ptr), stride, nfram, _stream_ptr(stream)))

    def results(self, stream=None):
        out = np.empty(self.n_inst, EBU_RESULT_DTYPE)
        _ck(lib().b200m_ebu_results(self.h, _np_ptr(out), _stream_ptr(stream)))
        return out

    def histogram(self, inst, stream=None):
        hm = np.empty(HIST_LEN, np.int32); hs = np.empty(HIST_LEN, np.int32)
        _ck(lib().b200m_ebu_histogram(self.h, inst, _np_ptr(hm), _np_ptr(hs), _stream_ptr(stream)))
        return hm, hs

    def coeffs(self):
        o = np.empty(7, np.float32)
        _ck(lib().b200m_ebu_coeffs(self.h, _np_ptr(o)))
        return o

    def state(self, inst, stream=None):
        z = np.empty((self.nchan, 4), np.float32); pw = np.empty(64, np.float32)
        fr = np.empty(1, np.float32); c = np.empty(4, np.int32)
        _ck(lib().b200m_ebu_state(self.h, inst, _np_ptr(z), _np_ptr(pw), _np_ptr(fr), _np_ptr(c), _stream_ptr(stream)))
        return z, pw, fr[0], c

    def mix_reduce(self, d_out, stream=None):
        """d_out: int32 CUDA tensor of MIX_WORDS elements."""
        _ck(lib().b200m_ebu_mix_reduce(self.h, C.c_void_p(d_out.data_ptr()), _stream_ptr(stream)))

    def mix_finish(self, d_mix, stream=None):
        out = np.empty(5, np.float32)
        _ck(lib().b200m_ebu_mix_finish(self.h, C.c_void_p(d_mix.data_ptr()), _np_ptr(out), _stream_ptr(stream)))
        return out


TPK_TRUEPEAK, TPK_KMETER = 1, 2
TP_MODE_PROCESS, TP_MODE_MAX = 0, 1
PREC_EXACT, PREC_FMA = 0, 1


class TruePeakKmeter(_Bank):
    """N x (LV2M::TruePeakdsp + LV2M::Kmeterdsp), one mono meter of each per channel
    (jmeters/truepeakdsp.h:28-61, jmeters/kmeterdsp.h:27-62; combined as in src/dr14.c:391-394)."""
    _destroy = "b200m_tpk_destroy"

    def __init__(self, n_chan, fsamp=48000.0, flags=TPK_TRUEPEAK | TPK_KMETER, device=0):
        super().__init__()
        self.n_chan, self.flags = n_chan, flags
        _ck(lib().b200m_tpk_create(C.byref(self.h), device, n_chan, fsamp, flags))

    def process(self, x, tp_mode=TP_MODE_PROCESS, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == self.n_chan
            _ck(lib().b200m_tpk_process_host(self.h, p, s, n, tp_mode))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == self.n_chan
            _ck(lib().b200m_tpk_process_device(self.h, p, s, n, tp_mode, _stream_ptr(stream)))

    def process_ptr(self, ptr, stride, nfram, tp_mode=TP_MODE_PROCESS, stream=None):
        _ck(lib().b200m_tpk_process_device(self.h, C.c_void_p(ptr), stride, nfram, tp_mode, _stream_ptr(stream)))

    def process_max(self, x, stream=None):
        self.process(x, TP_MODE_MAX, stream)

    def set_precision(self, mode):
        """PREC_EXACT (bit-identical floats, default) or PREC_FMA (fused FIR, readings within +-1e-4 dB)"""
        _ck(lib().b200m_tpk_set_precision(self.h, int(mode)))

    def read_device(self, stream=None):
        _ck(lib().b200m_tpk_read_device(self.h, _stream_ptr(stream)))

    def results(self, stream=None):
        out = np.empty(self.n_chan, TPK_RESULT_DTYPE)
        _ck(lib().b200m_tpk_results(self.h, _np_ptr(out), _stream_ptr(stream)))
        return out

    def read(self, stream=None):
        """read() of every meter + fetch: the per-run() sequence of dr14_run (src/dr14.c:425-430)."""
        self.read_device(stream)
        return self.results(stream)

    def reset(self, chan=-1, stream=None):
        _ck(lib().b200m_tpk_reset(self.h, chan, _stream_ptr(stream)))

    def coeffs(self):
        w = np.empty(4, np.float32); t = np.empty(120, np.float32); k = np.empty(2, np.float32)
        _ck(lib().b200m_tpk_coeffs(self.h, _np_ptr(w), _np_ptr(t), _np_ptr(k)))
        return w, t, k

    def state(self, stream=None):
        n = self.n_chan
        m, p, z1, z2 = (np.empty(n, np.float32) for _ in range(4))
        res = np.empty(n, np.int32); km = np.empty((n, 8), np.float32)
        _ck(lib().b200m_tpk_state(self.h, _np_ptr(m), _np_ptr(p), _np_ptr(z1), _np_ptr(z2), _np_ptr(res), _np_ptr(km), _stream_ptr(stream)))
        return dict(m=m, p=p, z1=z1, z2=z2, res=res, km=km)

    def debug_capture(self, enable=True):
        _ck(lib().b200m_tpk_debug_capture(self.h, int(enable)))

    def debug_upsampled(self, chan, n_out, stream=None):
        out = np.empty(n_out, np.float32)
        _ck(lib().b200m_tpk_debug_upsampled(self.h, chan, _np_ptr(out), n_out, _stream_ptr(stream)))
        return out


class Stcorrdsp(_Bank):
    """N x LV2M::Stcorrdsp (jmeters/stcorrdsp.h:27-55); channels 2i, 2i+1 = L, R of pair i."""
    _destroy = "b200m_cor_destroy"

    def __init__(self, n_inst, fsamp=48000, flp=2e3, tcf=0.3, device=0):
        super().__init__()
        self.n_inst = n_inst
        _ck(lib().b200m_cor_create(C.byref(self.h), device, n_inst, int(fsamp), flp, tcf))

    def process(self, x, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == 2 * self.n_inst
            _ck(lib().b200m_cor_process_host(self.h, p, s, n))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == 2 * self.n_inst
            _ck(lib().b200m_cor_process_device(self.h, p, s, n, _stream_ptr(stream)))

    def set_precision(self, mode):
        """PREC_EXACT: serial, bit-identical; PREC_FMA: time-parallel warp scan, correlation within 1e-5"""
        _ck(lib().b200m_cor_set_precision(self.h, int(mode)))

    def process_ptr(self, ptr, stride, nfram, stream=None):
        _ck(lib().b200m_cor_process_device(self.h, C.c_void_p(ptr), stride, nfram, _stream_ptr(stream)))

    def read(self, stream=None):
        out = np.empty(self.n_inst, np.float32)
        _ck(lib().b200m_cor_results(self.h, _np_ptr(out), _stream_ptr(stream)))
        return out

    def state(self, stream=None):
        s = np.empty((self.n_inst, 5), np.float32)
        _ck(lib().b200m_cor_state(self.h, _np_ptr(s), _stream_ptr(stream)))
        return s

    def coeffs(self):
        w = np.empty(2, np.float32)
        _ck(lib().b200m_cor_coeffs(self.h, _np_ptr(w)))
        return w


PPM_VU, PPM_IEC1, PPM_IEC2, PPM_MS = 0, 1, 2, 3


def design_ppm(kind, fsamp):
    w = np.empty(4, np.float32)
    _ck(lib().b200m_design_ppm(kind, fsamp, _np_ptr(w)))
    return w


class NeedleMeters(_Bank):
    """N x Vumeterdsp / Iec1ppmdsp / Iec2ppmdsp, or N stereo pairs x (Msppmdsp M, Msppmdsp S) (jmeters/*.cc)."""
    _destroy = "b200m_ppm_destroy"

    def __init__(self, n_units, kind, fsamp=48000.0, device=0):
        super().__init__()
        self.n_units, self.kind = n_units, kind
        self.rows = 2 * n_units if kind == PPM_MS else n_units
        self.n_meters = self.rows
        _ck(lib().b200m_ppm_create(C.byref(self.h), device, n_units, fsamp, kind))

    def set_gain(self, db_m, db_s):
        _ck(lib().b200m_ppm_set_gain(self.h, db_m, db_s))

    def process(self, x, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == self.rows
            _ck(lib().b200m_ppm_process_host(self.h, p, s, n))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == self.rows
            _ck(lib().b200m_ppm_process_device(self.h, p, s, n, _stream_ptr(stream)))

    def read(self, stream=None):
        _ck(lib().b200m_ppm_read_device(self.h, _stream_ptr(stream)))
        out = np.empty(self.n_meters, np.float32)
        _ck(lib().b200m_ppm_results(self.h, _np_ptr(out), _stream_ptr(stream)))
        return out

    def state(self, stream=None):
        s = np.empty((self.n_meters, 4), np.float32)
        _ck(lib().b200m_ppm_state(self.h, _np_ptr(s), _stream_ptr(stream)))
        return s


CTL_START, CTL_PAUSE, CTL_RESET, CTL_AVERAGE, CTL_WINDOWED = 1, 2, 3, 4, 5


class _StatBank(_Bank):
    _pfx = None

    def __init__(self, n_inst, rate=48000.0, device=0):
        super().__init__()
        self.n_inst = n_inst
        _ck(getattr(lib(), self._pfx + "create")(C.byref(self.h), device, n_inst, rate))

    def control(self, cmd, stream=None):
        _ck(getattr(lib(), self._pfx + "control")(self.h, cmd, _stream_ptr(stream)))

    def run(self, x, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == self.n_inst
            _ck(getattr(lib(), self._pfx + "run_host")(self.h, p, s, n))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == self.n_inst
            _ck(getattr(lib(), self._pfx + "run_device")(self.h, p, s, n, _stream_ptr(stream)))

    def run_ptr(self, ptr, stride, nfram, stream=None):
        _ck(getattr(lib(), self._pfx + "run_device")(self.h, C.c_void_p(ptr), stride, nfram, _stream_ptr(stream)))


class Bitmeter(_StatBank):
    """N x the bit-meter plugin's statistics (src/bitmeter.c:63-105,248-327)."""
    _destroy, _pfx = "b200m_bim_destroy", "b200m_bim_"

    def results(self, inst, stream=None):
        h = np.empty(584, np.int32); c = np.empty(5, np.int32); mm = np.empty(2, np.float32); it = C.c_int64(0)
        _ck(lib().b200m_bim_results(self.h, inst, _np_ptr(h), _np_ptr(c), _np_ptr(mm), C.byref(it), _stream_ptr(stream)))
        return h, c, mm, it.value


class SigDistHist(_StatBank):
    """N x the signal-distribution-histogram plugin's statistics (src/sigdistlv2.c:287-327)."""
    _destroy, _pfx = "b200m_sdh_destroy", "b200m_sdh_"

    def results(self, inst, stream=None):
        h = np.empty(361, np.int32); mp = np.empty(2, np.int32); av = np.empty(3, np.float64); it = C.c_int64(0)
        _ck(lib().b200m_sdh_results(self.h, inst, _np_ptr(h), _np_ptr(mp), _np_ptr(av), C.byref(it), _stream_ptr(stream)))
        return h, mp, av, it.value


DR14_RESULT_DTYPE = np.dtype([("v_rms", "<f4", 2), ("v_peak", "<f4", 2), ("m_peak", "<f4", 2), ("m_rms", "<f4", 2), ("dr", "<f4", 2),
                              ("dr_total", "<f4"), ("block_count", "<f4")])


class DR14(_Bank):
    """N x dr14_run (src/dr14.c:354-482): DR-14 mode (dr_mode=True) or TPnRMS (False); results = the plugin's output ports."""
    _destroy = "b200m_dr14_destroy"

    def __init__(self, n_inst, n_channels=2, rate=48000.0, dr_mode=True, device=0):
        super().__init__()
        self.n_inst, self.nchan = n_inst, n_channels
        _ck(lib().b200m_dr14_create(C.byref(self.h), device, n_inst, n_channels, rate, int(bool(dr_mode))))

    def run(self, x, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == self.n_inst * self.nchan
            _ck(lib().b200m_dr14_run_host(self.h, p, s, n))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == self.n_inst * self.nchan
            _ck(lib().b200m_dr14_run_device(self.h, p, s, n, _stream_ptr(stream)))

    def run_ptr(self, ptr, stride, nfram, stream=None):
        _ck(lib().b200m_dr14_run_device(self.h, C.c_void_p(ptr), stride, nfram, _stream_ptr(stream)))

    def reset(self, stream=None):
        _ck(lib().b200m_dr14_reset(self.h, _stream_ptr(stream)))

    def results(self, stream=None):
        out = np.empty(self.n_inst, DR14_RESULT_DTYPE)
        _ck(lib().b200m_dr14_results(self.h, _np_ptr(out), _stream_ptr(stream)))
        return out

    def histogram(self, inst, chan, stream=None):
        h = np.empty(8000, np.uint32)
        _ck(lib().b200m_dr14_histogram(self.h, inst, chan, _np_ptr(h), _stream_ptr(stream)))
        return h


class Spectr30(_Bank):
    """N x the spectr30 plugin (src/spectrumlv2.c:73-257): ports 0..59 per instance."""
    _destroy = "b200m_spec_destroy"

    def __init__(self, n_inst, nchan=2, rate=48000.0, device=0):
        super().__init__()
        self.n_inst, self.nchan = n_inst, nchan
        _ck(lib().b200m_spec_create(C.byref(self.h), device, n_inst, nchan, rate))

    def process(self, x, speed=1.0, reset=-4.0, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == self.n_inst * self.nchan
            _ck(lib().b200m_spec_process_host(self.h, p, s, n, speed, reset))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == self.n_inst * self.nchan
            _ck(lib().b200m_spec_process_device(self.h, p, s, n, speed, reset, _stream_ptr(stream)))

    def set_precision(self, mode):
        """PREC_EXACT: ports bit-identical to the reference; PREC_FMA: fused multiply-adds, band levels within +-1e-4 dB"""
        _ck(lib().b200m_spec_set_precision(self.h, int(mode)))

    def process_ptr(self, ptr, stride, nfram, speed=1.0, reset=-4.0, stream=None):
        _ck(lib().b200m_spec_process_device(self.h, C.c_void_p(ptr), stride, nfram, speed, reset, _stream_ptr(stream)))

    def read(self, stream=None):
        out = np.empty((self.n_inst, 60), np.float32)
        _ck(lib().b200m_spec_results(self.h, _np_ptr(out), _stream_ptr(stream)))
        return out

    def state(self, inst, stream=None):
        z = np.empty((30, 6, 2), np.float64); v = np.empty(30, np.float32); m = np.empty(30, np.float32)
        _ck(lib().b200m_spec_state(self.h, inst, _np_ptr(z), _np_ptr(v), _np_ptr(m), _stream_ptr(stream)))
        return z, v, m

    def coeffs(self):
        W = np.empty((30, 6, 6), np.float64)
        _ck(lib().b200m_spec_coeffs(self.h, _np_ptr(W)))
        return W


class Phasewheel(_Bank):
    """N x (2 x FFTAnalysis + phasewheel process_audio) (gui/fft.c:208-361, gui/phasewheel.c:1307-1342)."""
    _destroy = "b200m_pw_destroy"

    def __init__(self, n_inst, fft_bins=1024, rate=48000.0, device=0):
        super().__init__()
        self.n_inst, self.bins = n_inst, fft_bins
        _ck(lib().b200m_pw_create(C.byref(self.h), device, n_inst, fft_bins, rate))

    def process(self, x, db_thresh=1e-6, stream=None):
        fired = C.c_int(0)
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == 2 * self.n_inst
            _ck(lib().b200m_pw_process_host(self.h, p, s, n, db_thresh, C.byref(fired)))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == 2 * self.n_inst
            _ck(lib().b200m_pw_process_device(self.h, p, s, n, db_thresh, C.byref(fired), _stream_ptr(stream)))
        return fired.value

    def process_ptr(self, ptr, stride, nfram, db_thresh=1e-6, stream=None):
        fired = C.c_int(0)
        _ck(lib().b200m_pw_process_device(self.h, C.c_void_p(ptr), stride, nfram, db_thresh, C.byref(fired), _stream_ptr(stream)))
        return fired.value

    def debug_capture(self, enable=True):
        """keep ft->power / ft->phase of both channels of every analysis (needed by raw())"""
        _ck(lib().b200m_pw_debug_capture(self.h, int(enable)))

    def attach_cor(self, cor):
        """fused feed: process*() also runs `cor` (a Stcorrdsp bank of n_inst pairs) on the same block, reading the input once"""
        _ck(lib().b200m_pw_attach_cor(self.h, cor.h if cor is not None else None))
        self._cor = cor

    def set_mode(self, mode):
        """0: phasewheel process_audio; 1: stereoscope process_audio (read() then returns lr[] as `phase`)"""
        _ck(lib().b200m_pw_set_mode(self.h, int(mode)))

    def read(self, stream=None):
        ph = np.empty((self.n_inst, self.bins), np.float32); lv = np.empty((self.n_inst, self.bins), np.float32)
        pk = np.empty(self.n_inst, np.float32)
        _ck(lib().b200m_pw_results(self.h, _np_ptr(ph), _np_ptr(lv), _np_ptr(pk), _stream_ptr(stream)))
        return ph, lv, pk

    def raw(self, inst, stream=None):
        a = [np.empty(self.bins, np.float32) for _ in range(4)]
        _ck(lib().b200m_pw_raw(self.h, inst, *[_np_ptr(v) for v in a], _stream_ptr(stream)))
        return a


class EBUr128(_Bank):
    """N x the EBUr128 plugin's audio cycle (ebur128_run, src/ebulv2.cc:341-367): EBU R128 + optional dBTP."""
    _destroy = "b200m_r128_destroy"
    START, PAUSE, RESET = 1, 2, 3

    def __init__(self, n_inst, fsamp=48000.0, dbtp_enable=True, device=0):
        super().__init__()
        self.n_inst = n_inst
        _ck(lib().b200m_r128_create(C.byref(self.h), device, n_inst, fsamp, int(dbtp_enable)))
        self.ebu = Ebu_r128_proc.__new__(Ebu_r128_proc)
        self.ebu.h = _v(lib().b200m_r128_ebu(self.h)); self.ebu.n_inst = n_inst; self.ebu.nchan = 2
        self.ebu._destroy = None

    def close(self):
        if getattr(self, "ebu", None) is not None:
            self.ebu.h = _v()
        super().close()

    def control(self, cmd, inst=-1, stream=None):
        _ck(lib().b200m_r128_control(self.h, inst, cmd, _stream_ptr(stream)))

    def run(self, x, stream=None):
        if isinstance(x, np.ndarray) or not x.is_cuda:
            p, s, rows, n = _host_planar(x)
            assert rows == 2 * self.n_inst
            _ck(lib().b200m_r128_run_host(self.h, p, s, n))
        else:
            p, s, rows, n = _dev_ptr(x)
            assert rows == 2 * self.n_inst
            _ck(lib().b200m_r128_run_device(self.h, p, s, n, _stream_ptr(stream)))

    def run_ptr(self, ptr, stride, nfram, stream=None, host=False):
        if host:
            _ck(lib().b200m_r128_run_host(self.h, C.c_void_p(ptr), stride, nfram))
        else:
            _ck(lib().b200m_r128_run_device(self.h, C.c_void_p(ptr), stride, nfram, _stream_ptr(stream)))

    def run_pcm(self, x, interleaved, stream=None):
        """one cycle on integer or float PCM, converted on the GPU: planar [2N, nfram] or interleaved [N, nfram, 2]; int16,
        int32, float32, or uint8 [..., 3] for packed 24-bit.  numpy / CPU tensors take the host path, CUDA tensors the device path."""
        p, fmt, stride, nfram, nseg, dev = _pcm_layout(x, interleaved, 2)
        assert nseg == (self.n_inst if interleaved else 2 * self.n_inst), "want %d %s" % (
            self.n_inst if interleaved else 2 * self.n_inst, "instances" if interleaved else "rows")
        self.run_pcm_ptr(p, fmt, stride, nfram, stream, host=not dev)

    def run_pcm_ptr(self, ptr, fmt, stride, nfram, stream=None, host=False):
        """b200m_r128_run_host_pcm / _run_device_pcm on a raw pointer; fmt = PCM_{F32,S16,S24,S32} | PCM_{PLANAR,INTERLEAVED}"""
        if host:
            _ck(lib().b200m_r128_run_host_pcm(self.h, C.c_void_p(ptr), fmt, stride, nfram))
        else:
            _ck(lib().b200m_r128_run_device_pcm(self.h, C.c_void_p(ptr), fmt, stride, nfram, _stream_ptr(stream)))

    def results(self, stream=None, out=None, tp=None):
        out = np.empty(self.n_inst, EBU_RESULT_DTYPE) if out is None else out
        tp = np.empty(self.n_inst, np.float32) if tp is None else tp
        _ck(lib().b200m_r128_results(self.h, _np_ptr(out), _np_ptr(tp), _stream_ptr(stream)))
        return out, tp

    def snapshot(self, stream=None):
        """the whole bank state as bytes (checkpoint)"""
        n = lib().b200m_r128_snapshot_size(self.h)
        buf = np.empty(n, np.uint8)
        _ck(lib().b200m_r128_snapshot(self.h, _np_ptr(buf), n, _stream_ptr(stream)))
        return buf

    def restore(self, blob, stream=None):
        blob = np.ascontiguousarray(blob, np.uint8)
        _ck(lib().b200m_r128_restore(self.h, _np_ptr(blob), blob.size, _stream_ptr(stream)))

    def set_dbtp(self, enable):
        """self->dbtp_enable (src/ebulv2.cc:316-317): takes effect with the next run"""
        _ck(lib().b200m_r128_set_dbtp(self.h, int(bool(enable))))

    def set_precision(self, mode):
        """precision of the dBTP FIR (PREC_EXACT / PREC_FMA); the EBU R128 part is always exact"""
        _ck(lib().b200m_r128_set_precision(self.h, int(mode)))

    def histogram(self, inst, stream=None):
        m = np.empty(751, np.int32); s = np.empty(751, np.int32)
        _ck(lib().b200m_r128_histogram(self.h, int(inst), _np_ptr(m), _np_ptr(s), _stream_ptr(stream)))
        return m, s
