"""CPU: the C-ABI library loads, exports every symbol include/b200meters.h declares, designs its coefficients
bitwise like the reference, and refuses to work without a GPU (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import _oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def u32(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_library_exports_every_declared_symbol():
    import meters_lv2_b200 as B
    hdr = open(os.path.join(ROOT, "include", "b200meters.h")).read()
    declared = set(re.findall(r"\b(b200m_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 55
    L = C.CDLL(B.LIB_PATH)
    missing = [n for n in sorted(declared) if not hasattr(L, n)]
    assert not missing, missing
    assert B.missing_exports() == []
    assert set(B.EXPORTS) == declared, sorted(set(B.EXPORTS) ^ declared)
    assert B.lib().b200m_abi_version() == 1


def test_no_cpu_fallback_without_device():
    import torch
    import meters_lv2_b200 as B
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert B.lib().b200m_device_count() == 0
    for ctor in (lambda: B.Ebu_r128_proc(2), lambda: B.TruePeakKmeter(2), lambda: B.Stcorrdsp(2),
                 lambda: B.Spectr30(2), lambda: B.Phasewheel(2)):
        with pytest.raises(B.B200MError, match="no CUDA device"):
            ctor()


def test_argument_errors_are_codes_not_crashes():
    import meters_lv2_b200 as B
    L = B.lib()
    assert L.b200m_ebu_create(None, 0, 1, 2, 48000.0) == -1
    h = C.c_void_p()
    assert L.b200m_ebu_create(C.byref(h), 0, 0, 2, 48000.0) == -1          # n_inst = 0
    assert L.b200m_ebu_create(C.byref(h), 0, 4, 7, 48000.0) == -1          # nchan outside 1..5
    assert L.b200m_pw_create(C.byref(h), 0, 4, 1000, 48000.0) == -1        # not a power of two
    assert L.b200m_ebu_process_device(None, None, 0, 0, None) == -1
    assert b"NULL" in L.b200m_last_error()
    assert L.b200m_ebu_destroy(None) == 0


def test_lv2_descriptor_table_and_instantiate_failures(reftape):
    """the LV2 facade enumerates all 38 URIs of the reference (src/meters.cc:745-792) and, like the reference, answers
    instantiate() with NULL when it cannot run: no urid:map feature for the atom plugins, no GPU for any"""
    import torch
    import meters_lv2_b200 as B
    from test_lv2_shim_gpu import Feature, _feats, descriptors
    d, lib = descriptors(B.LIB_PATH)
    uris = set(d)
    assert len(uris) == 38
    for u in ("EBUr128", "dr14stereo", "TPnRMSmono", "SigDistHist", "bitmeter", "phasewheel", "stereoscope", "surround8", "K20stereo", "BBCM6", "goniometer"):
        assert u in uris, u
    assert uris == set(reftape.ref(lambda: sorted(descriptors(O.PATHS["reference"])[0])))
    none = (C.POINTER(Feature) * 1)(None)
    for u in ("EBUr128", "dr14mono", "SigDistHist", "bitmeter", "phasewheel", "goniometer"):
        assert not d[u].contents.instantiate(d[u], 48000.0, b"", none), u           # urid:map missing -> NULL
    if not torch.cuda.is_available():
        for u in ("EBUr128", "K20stereo", "COR", "spectr30stereo", "surround5", "goniometer"):
            assert not d[u].contents.instantiate(d[u], 48000.0, b"", _feats), u     # no device, no CPU fallback -> NULL


@pytest.mark.parametrize("fs", [48000.0, 44100.0, 96000.0, 88200.0, 192000.0])
def test_host_design_bitwise_equals_oracle(fs):
    import meters_lv2_b200 as B
    assert np.array_equal(u32(B.design_ebu(fs)), u32(O.Ebu(1, 2, fs).coeffs()))
    w, t, k = B.design_tpk(fs)
    ow, ot = O.TruePeak(1, fs).coeffs()
    om, oh = O.Kmeter(1, fs).coeffs()
    assert np.array_equal(u32(w), u32(ow)) and np.array_equal(u32(t), u32(ot))
    assert u32(k[:1])[0] == u32(np.float32(om))[()] and int(k[1]) == oh
    assert np.array_equal(u32(B.design_cor(fs)), u32(O.Stcorr(1, fs).coeffs()))
    for k in range(4):
        assert np.array_equal(u32(B.design_ppm(k, fs)), u32(O.Needle(1, k, fs).coeffs())), k
    W = B.design_spec(fs)
    R = O.Spectr30(1, 2, fs).coeffs()
    assert np.array_equal(W.view(np.uint64), R.view(np.uint64))
    # stage 0 carries the gain: b1 = 2*b0, b2 = b0 ; stages 1..5 are (1, +-2, 1)
    assert np.array_equal(W[:, 0, 4], 2 * W[:, 0, 3]) and np.array_equal(W[:, 0, 5], W[:, 0, 3])
    assert (W[:, 1:, 3] == 1).all() and (np.abs(W[:, 1:, 4]) == 2).all() and (W[:, 1:, 5] == 1).all()


def test_appendix_a_constants_48k():
    """SURVEY.md App. A (oracle-derived constants at 48 kHz)."""
    import meters_lv2_b200 as B
    e = B.design_ebu(48000.0)
    assert np.allclose(e, [1.5351752, -2.69206738, 1.19870186, -1.69091594, 0.732725799, 0.00995242409, 2.47953594e-05], rtol=2e-7)
    w, t, k = B.design_tpk(48000.0)
    assert np.allclose(w, [0.020833334, 0.0895833299, 0.999963522, 0.501999974], rtol=1e-7)
    assert t[23] == 1.0 and abs(t[47] - 0.899852) < 1e-6 and abs(t[71] - 0.635306) < 1e-6 and abs(t[95] - 0.298714) < 1e-6
    assert abs(k[0] - 0.000202499999) < 1e-12 and k[1] == 24000
    assert np.allclose(B.design_cor(48000), [0.261666656, 6.94444389e-05], rtol=1e-7)
    W = B.design_spec(48000.0)
    # the survey's probe printed the 1 kHz band to ~1e-7 relative only (its band edges were computed slightly
    # differently); the bitwise pin is test_host_design_bitwise_equals_oracle above
    assert abs(W[16, 0, 1] / -1.9702830368451048 - 1) < 1e-6 and abs(W[16, 0, 3] / 1.1434061583804783e-11 - 1) < 1e-3
