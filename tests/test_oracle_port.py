"""CPU: pins the oracle.  (1) the port (oracle/oracle_port.cc, this repo's restatement) must equal the
reference build (oracle/_ref, the unmodified reference sources) bit for bit on seeded streams;
(2) both must reproduce the committed golden vectors (tests/golden/*.npz, generated from oracle/_ref by
tests/golden/make_golden.py) and the survey's known-answer values (SURVEY.md App. C).  Where oracle/_ref is not built, the
reference side of (1) is replayed from its recording (tests/_reftape.py)."""
import os

import numpy as np
import pytest

import _oracle as O
import _reftape as R
import _signals as S

HAVE_REF = O.available("reference")
HAVE_PORT = O.available("port")
needs_port = pytest.mark.skipif(not HAVE_PORT, reason="run `make -C oracle port`")
BLOCKS = [1024] * 30 + [64] * 8 + [480] * 4 + [8192, 1, 3, 1023, 2401, 4799]


def u32(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _blocks(x, blocks):
    pos = 0
    for n in blocks:
        yield np.ascontiguousarray(x[:, pos:pos + n])
        pos += n


@needs_port
@pytest.mark.parametrize("nchan", [1, 2])
def test_ebu_port_equals_reference(nchan, reftape):
    t = reftape
    x = S.white(6 * nchan, sum(BLOCKS) + 1024 * 280, seed=101)
    a, b = t.obj(lambda: O.Ebu(6, nchan, kind="reference")), O.Ebu(6, nchan, kind="port")
    assert np.array_equal(u32(t.ref(lambda: a.coeffs())), u32(b.coeffs()))
    a.integr("start"); b.integr("start")
    for blk in _blocks(x, BLOCKS + [1024] * 280):
        a.process(blk); b.process(blk)
    assert np.array_equal(u32(t.ref(lambda: a.read())), u32(b.read()))
    for i in range(6):
        ha, hb = t.refs(lambda: a.hist(i), 3), b.hist(i)
        assert all(np.array_equal(p, q) for p, q in zip(ha, hb))
        sa, sb = t.refs(lambda: a.state(i), 4), b.state(i)
        assert np.array_equal(u32(sa[0]), u32(sb[0])) and np.array_equal(u32(sa[1]), u32(sb[1])) and list(sa[3]) == list(sb[3])


@needs_port
def test_truepeak_kmeter_port_equals_reference(reftape):
    t = reftape
    x = S.nasty(7, sum(BLOCKS), seed=102)
    wa, ta = t.refs(lambda: O.TruePeak(1, kind="reference").coeffs(), 2); wb, tb = O.TruePeak(1, kind="port").coeffs()
    assert np.array_equal(u32(wa), u32(wb)) and np.array_equal(u32(ta), u32(tb))
    for mode in (0, 1):
        a, b = t.obj(lambda: O.TruePeak(7, kind="reference")), O.TruePeak(7, kind="port")
        ka, kb = t.obj(lambda: O.Kmeter(7, kind="reference")), O.Kmeter(7, kind="port")
        for i, blk in enumerate(_blocks(x, BLOCKS)):
            a.process(blk, mode); b.process(blk, mode); ka.process(blk); kb.process(blk)
            if i % 3 == 0:
                ra, rb = t.ref(lambda: a.read()), b.read()
                assert np.array_equal(u32(ra[0]), u32(rb[0])) and np.array_equal(u32(ra[1]), u32(rb[1]))
                qa, qb = t.ref(lambda: ka.read()), kb.read()
                assert np.array_equal(u32(qa[0]), u32(qb[0])) and np.array_equal(u32(qa[1]), u32(qb[1]))
        assert all(np.array_equal(u32(p), u32(q)) for p, q in zip(t.ref(lambda: a.peek()[:4]), b.peek()[:4]))
        assert np.array_equal(u32(t.ref(lambda: ka.peek())), u32(kb.peek()))
    y = S.white(1, 5000, seed=3)[0]
    assert t.digest(lambda: u32(O.tp_upsample(y, kind="reference"))) == R.digest(u32(O.tp_upsample(y, kind="port")))


@needs_port
def test_stcorr_port_equals_reference(reftape):
    t = reftape
    x = S.nasty(10, sum(BLOCKS), seed=103)
    a, b = t.obj(lambda: O.Stcorr(5, kind="reference")), O.Stcorr(5, kind="port")
    assert np.array_equal(u32(t.ref(lambda: a.coeffs())), u32(b.coeffs()))
    for blk in _blocks(x, BLOCKS):
        a.process(blk); b.process(blk)
        assert np.array_equal(u32(t.ref(lambda: a.read())), u32(b.read()))
    assert np.array_equal(u32(t.ref(lambda: a.peek())), u32(b.peek()))


@needs_port
@pytest.mark.parametrize("nchan,rate", [(2, 48000.0), (1, 44100.0)])
def test_spectr_port_equals_reference(nchan, rate, reftape):
    t = reftape
    x = S.white(2 * nchan, 1024 * 6 + 777, seed=104)
    a, b = t.obj(lambda: O.Spectr30(2, nchan, rate, kind="reference")), O.Spectr30(2, nchan, rate, kind="port")
    assert np.array_equal(t.ref(lambda: a.coeffs()).view(np.uint64), b.coeffs().view(np.uint64))
    for i, blk in enumerate(_blocks(x, [1024] * 6 + [777])):
        spd = 1.0 if i < 3 else 4.0
        a.process(blk, spd, -4.0); b.process(blk, spd, -4.0)
        pa, pb = t.ref(lambda: a.read()), b.read()
        assert np.array_equal(u32(pa[:, :30]), u32(pb[:, :30]))
        ok = pa[:, 30:] > -500
        assert np.array_equal(u32(pa[:, 30:][ok]), u32(pb[:, 30:][ok]))
    za, zb = t.refs(lambda: a.state(1), 3), b.state(1)
    assert np.array_equal(za[0].view(np.uint64), zb[0].view(np.uint64)) and np.array_equal(u32(za[1]), u32(zb[1]))


@needs_port
@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_needle_meters_port_equals_reference(kind, reftape):
    t = reftape
    n = 5
    rows = 2 * n if kind == 3 else n
    x = S.nasty(rows, sum(BLOCKS), seed=106 + kind) * np.float32(3.0)
    a, b = t.obj(lambda: O.Needle(n, kind, oracle="reference")), O.Needle(n, kind, oracle="port")
    assert np.array_equal(u32(t.ref(lambda: a.coeffs())), u32(b.coeffs()))
    if kind == 3:
        a.set_gain(-6, 14); b.set_gain(-6, 14)
    for i, blk in enumerate(_blocks(x, BLOCKS)):
        a.process(blk); b.process(blk)
        if i % 2:
            assert np.array_equal(u32(t.ref(lambda: a.read())), u32(b.read()))
    assert np.array_equal(u32(t.ref(lambda: a.peek())), u32(b.peek()))


@needs_port
def test_bitmeter_and_sigdist_port_equals_reference_plugins(reftape):
    """the reference side runs the plugins' own LV2 run() (src/meters.cc compiled unmodified against oracle/lv2stub)"""
    t = reftape
    x = S.nasty(6, sum(BLOCKS), seed=111)
    x[1] *= np.float32(1e-39); x[2] *= np.float32(3.0); x[3] = 0
    for avg in (1, 0):
        a, b = t.obj(lambda: O.Bitmeter(6, oracle="reference")), O.Bitmeter(6, oracle="port")
        a.mode(avg); b.mode(avg)
        for blk in _blocks(x, BLOCKS):
            a.process(blk); b.process(blk)
            for i in range(6):
                r, rb = t.obj(lambda: a.read(i)), b.read(i)
                ra = [t.digest(lambda: r[0])] + t.refs(lambda: r[1:], 3)         # the 584-bin histogram by its digest
                assert ra[0] == R.digest(rb[0]) and np.array_equal(ra[1], rb[1]) and ra[3] == rb[3]
                assert np.array_equal(ra[2].view(np.uint32), rb[2].view(np.uint32))
    a, b = t.obj(lambda: O.SigDist(6, oracle="reference")), O.SigDist(6, oracle="port")
    a.integrate(); b.integrate()
    for blk in _blocks(x, BLOCKS):
        a.process(blk); b.process(blk)
    for i in range(6):
        ra, rb = t.refs(lambda: a.read(i), 4), b.read(i)
        assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1]) and ra[3] == rb[3]
        assert np.array_equal(ra[2].view(np.uint64), rb[2].view(np.uint64))


@needs_port
@pytest.mark.parametrize("nch,dr_mode,rate,block", [(2, True, 48000.0, 8192), (1, True, 44100.0, 1000), (2, False, 48000.0, 1024)])
def test_dr14_port_equals_reference_plugins(nch, dr_mode, rate, block, reftape):
    """restatement of dr14_run / dr14_calc_rms_score vs the reference's dr14 / TPnRMS plugins run through their own LV2 run()"""
    n_inst = 3
    nb = int(rate * 22 / block) if dr_mode else 30
    t = np.arange(nb * block) / rate
    env = (0.15 + 0.85 * np.abs(np.sin(2 * np.pi * t / 5.3))).astype(np.float32)
    x = (S.white(n_inst * nch, nb * block, seed=123) * env * np.float32(2.0)).astype(np.float32)
    x[0, 5 * block + 7] = np.nan                                # one poisoned window
    x[nch:2 * nch] *= np.float32(1e-6)                           # instance 1 stays below the silence gate
    a, b = reftape.obj(lambda: O.Dr14(n_inst, nch, rate, dr_mode, kind="reference")), O.Dr14(n_inst, nch, rate, dr_mode, kind="port")
    for k in range(nb):
        blk = np.ascontiguousarray(x[:, k * block:(k + 1) * block])
        a.process(blk); b.process(blk)
        if k == nb // 2 + 3:
            a.reset(); b.reset()
        ra, rb = reftape.ref(lambda: a.read()), b.read()
        same = (u32(ra) == u32(rb)) | (np.isnan(ra) & np.isnan(rb))
        assert same.all(), (k, ra[~same], rb[~same])
    if dr_mode:
        assert ra[0, 11] > 0 and ra[1, 11] == 0                  # scored windows on the loud instance only


@needs_port
@pytest.mark.parametrize("bins", [64, 512, 1024, 4096, 6144, 8192])
def test_port_phasewheel_against_numpy_fft(bins):
    """the FFT restatement is pinned to an INDEPENDENT float64 FFT (numpy / pocketfft) for every size the GUI offers
    (gui/phasewheel.c:1108-1116): powers AND phases, i.e. the half-complex layout and the sign convention of gui/fft.c:163-180."""
    import _fftref as F
    N = 2 * bins
    total = max(3 * N, 6000)
    x = S.white(2, total, seed=105)
    x[1, :] = 0.5 * S.sine(total, 48000.0 * 37 / N, phase=0.7)         # a bin-centred tone with a known phase on the right channel
    p = O.Phasewheel(1, bins, kind="port")
    pos, fired_end = 0, -1
    for n in [500] * (total // 500):
        if p.process(np.ascontiguousarray(x[:, pos:pos + n])):
            fired_end = pos + n
        pos += n
    assert fired_end >= N
    X, P, PH = F.spectra(x[:, fired_end - N:fired_end])
    powL, powR, phL, phR = p.raw(0)
    for ch, (pw, ph) in enumerate(((powL, phL), (powR, phR))):
        rel, db, dph = F.compare(pw, ph, X[ch])
        assert rel <= 2e-7 and db <= 1e-5 and dph <= 1e-6, (bins, ch, rel, db, dph)     # double DFT vs double FFT: float32 storage only
    assert powL[0] == np.float32(X[0, 0].real) ** 2 or abs(powL[0] - X[0, 0].real ** 2) <= 1e-6 * max(1e-30, X[0, 0].real ** 2)
    assert abs(phR[37] - np.angle(X[1, 37])) < 1e-5


@needs_port
def test_known_answers_survey_appendix_c():
    """SURVEY.md App. C: values the survey generated from the reference build (LCG noise, 4688 x 1024)."""
    nb = 4688
    x = S.lcg_stereo(1024 * nb)
    for kind in (["port", "reference"] if HAVE_REF else ["port"]):
        k = O.Kmeter(1, kind=kind); c = O.Stcorr(1, kind=kind); t = O.TruePeak(1, kind=kind)
        e = O.Ebu(1, kind=kind); e.integr("start")
        pmax = 0.0
        for blk in _blocks(x, [1024] * nb):
            e.process(blk); k.process(blk[:1]); c.process(blk); t.process(blk[:1])
            rms, pk = k.read(); m, p = t.read(); pmax = max(pmax, float(p[0]))
        r = e.read()[0]
        want = np.array([-10.673171, -10.666748, -10.689788, -20.689789], np.float32)
        assert np.allclose(r[[0, 2, 4, 5]], want, atol=2e-6, rtol=0), r
        hm, hs, cnt = e.hist(0)
        assert cnt[0] == 1000 and cnt[1] == 200
        assert np.float32(rms[0]) == np.float32(0.20495217) and np.float32(pk[0]) == np.float32(0.24985489)
        assert abs(float(c.read()[0]) - (-0.02344654)) < 1e-8
        assert abs(pmax - 0.50329632) < 1e-8


GOLD = os.path.join(os.path.dirname(__file__), "golden", "golden_v1.npz")


@needs_port
@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden vectors not generated")
@pytest.mark.parametrize("kind", ["port"] + (["reference"] if HAVE_REF else []))
def test_golden_vectors(kind):
    import golden.make_golden as G
    got = G.compute(kind)
    ref = np.load(GOLD)
    assert set(got) == set(ref.files)
    for k in ref.files:
        a, b = got[k], ref[k]
        if k.startswith("pw_"):                               # FFT path: double DFT, still deterministic on one libm
            assert np.allclose(a, b, rtol=1e-5, atol=1e-7), k
        elif k.startswith("spec_maxports"):
            ok = b > -500
            assert np.array_equal(a[ok].view(np.uint32), b[ok].view(np.uint32)), k
        else:
            assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
