"""Pins the CPU restatement (oracle/world_oracle.cpp) against the golden vectors generated from the
unmodified reference, and against the compiled reference itself on synthetic speech.
The restatement uses an independent FFT and libstdc++'s sort, so agreement is to rounding
(SURVEY.md App. B4b: <= 1e-10 on sp), not bit-exact."""
import os
import subprocess

import numpy as np
import pytest

import test_parity_common as pc
from refworld import RefWorld, ORACLE_LIB, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def port():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "libworld_oracle.so"])
    return RefWorld(ORACLE_LIB)


def test_port_matches_golden_vectors(port, golden):
    x, fs = pc.wav_from_golden(golden)
    t = golden["time_axis"]
    sm = port.stonemask(x, fs, t, golden["f0_dio"])
    assert rel_err(sm, golden["f0_stonemask"]).max() < 1e-9
    f0 = golden["f0_stonemask"]
    sp = port.cheaptrick(x, fs, t, f0)
    ap = port.d4c(x, fs, t, f0, int(golden["fft_size"]))
    assert rel_err(sp, golden["sp"]).max() < 1e-8
    assert rel_err(ap, golden["ap"]).max() < 1e-8


def test_port_matches_reference_on_synthetic(port, ref):
    from synth import synth_batch
    for fs, n, seed in ((16000, 12000, 51), (48000, 14400, 52)):
        x = synth_batch([seed], fs, n).numpy()[0]
        t, f0 = ref.dio(x, fs)
        f0r = ref.stonemask(x, fs, t, f0)
        assert rel_err(port.stonemask(x, fs, t, f0), f0r).max() < 1e-9
        o = ref.cheaptrick_option(fs)
        assert rel_err(port.cheaptrick(x, fs, t, f0r, o), ref.cheaptrick(x, fs, t, f0r, o)).max() < 1e-8
        assert rel_err(port.d4c(x, fs, t, f0r, o.fft_size), ref.d4c(x, fs, t, f0r, o.fft_size)).max() < 1e-8


def test_port_sizing_helpers(port, ref):
    for fs in (8000, 16000, 22050, 44100, 48000):
        assert port.cheaptrick_option(fs).fft_size == ref.cheaptrick_option(fs).fft_size
        assert port.frames(fs, 12345) == ref.frames(fs, 12345)


def test_port_codec_matches_golden_and_reference(port, ref, golden):
    """rows f2 / f3: the restated codec and PCM conversion against the reference's outputs."""
    import ctypes as C
    fs, fft, dims = int(golden["fs"]), int(golden["fft_size"]), int(golden["coded_dims"])
    assert port.has_codec and port.number_of_aperiodicities(fs) == golden["coded_ap"].shape[1]
    csp = port.code_spectral_envelope(golden["sp"], fs, fft, dims)
    cap = port.code_aperiodicity(golden["ap"], fs, fft)
    pc.assert_close_signed(csp, golden["coded_sp"], "port CodeSpectralEnvelope", tol=1e-9)
    pc.assert_close_signed(cap, golden["coded_ap"], "port CodeAperiodicity", tol=1e-9)
    assert rel_err(port.decode_spectral_envelope(golden["coded_sp"], fs, fft, dims)[::4], golden["decoded_sp_rows"]).max() < 1e-9
    assert rel_err(port.decode_aperiodicity(golden["coded_ap"], fs, fft)[::4], golden["decoded_ap_rows"]).max() < 1e-9
    for fs2, fft2, d in ((16000, 1024, 60), (48000, 2048, 24), (8000, 512, 129)):
        rng = np.random.default_rng(fs2)
        sp = np.exp(rng.normal(size=(5, fft2 // 2 + 1)) * 3 - 8)
        want = ref.code_spectral_envelope(sp, fs2, fft2, d)
        pc.assert_close_signed(port.code_spectral_envelope(sp, fs2, fft2, d), want, "port code sp", tol=1e-9)
        assert rel_err(port.decode_spectral_envelope(want, fs2, fft2, d), ref.decode_spectral_envelope(want, fs2, fft2, d)).max() < 1e-9
        assert port.number_of_aperiodicities(fs2) == ref.number_of_aperiodicities(fs2)
    pcm = np.ascontiguousarray(golden["pcm"])
    x = np.zeros(len(pcm))
    port.lib.OraclePcmToDouble(pcm.ctypes.data_as(C.c_void_p), 16, len(pcm), x.ctypes.data_as(C.c_void_p))
    assert np.array_equal(x, pc.wav_from_golden(golden)[0])


def test_port_dio_matches_golden_and_reference(port, ref, golden):
    """The time-domain restatement of Dio (no FFT anywhere) against the reference's FFT-based one."""
    assert port.has_dio
    x, fs = pc.wav_from_golden(golden)
    t, f0 = port.dio(x, fs)
    assert np.array_equal(t, golden["time_axis"])
    assert rel_err(f0, golden["f0_dio"]).max() < 1e-9
    o = port.dio_option(); o.f0_floor = 40.0
    assert rel_err(port.dio(x, fs, o)[1], golden["f0_dio_floor40"]).max() < 1e-9
    from synth import synth_batch
    for fs2, n, seed, speed in ((16000, 16000, 71, 1), (44100, 22050, 72, 11), (48000, 24000, 73, 4)):
        xs = synth_batch([seed], fs2, n).numpy()[0]
        po = port.dio_option(); po.speed = speed
        ro = ref.dio_option(); ro.speed = speed
        tp, fp = port.dio(xs, fs2, po)
        tr, fr = ref.dio(xs, fs2, ro)
        assert np.array_equal(tp, tr)
        # time-domain filtering here, whole-utterance FFT convolution there -- plus the ripple of the reference's
        # spectral mirroring loop written out (see Dio in oracle/world_oracle.cpp): without it the decimated
        # cases sat 2e-9 (here) to 2e-2 (speed 10..12 at 8..16 kHz) from the reference
        r = rel_err(fp, fr)
        assert r.max() < 1e-9, (fs2, speed, r.max())
        assert (fr > 0).sum() > 20
        y1 = np.zeros(len(xs)); y2 = np.zeros(len(xs))
        if speed > 1:   # the restated decimate() alone is bit-identical to the reference's
            import ctypes as C
            y1 = ref.decimate(xs, speed)
            port.lib.OracleDecimate(xs.ctypes.data_as(C.c_void_p), len(xs), speed, y2.ctypes.data_as(C.c_void_p))
            assert np.ma.allequal(y1, y2)


def test_port_harvest_matches_golden_and_reference(port, ref, golden):
    """The restated Harvest (time-domain band-pass FIRs, own FFT for the refinement) against the goldens and
    the compiled reference: all frame periods / rates of the parity matrix, no V/UV flip allowed."""
    assert port.has_harvest
    x, fs = pc.wav_from_golden(golden)
    t, f0 = port.harvest(x, fs)
    assert np.array_equal(t, golden["time_axis"])
    assert rel_err(f0, golden["f0_harvest"]).max() < 1e-9
    o = port.harvest_option(); o.f0_floor = 40.0
    assert rel_err(port.harvest(x, fs, o)[1], golden["f0_harvest_floor40"]).max() < 1e-9
    from synth import synth_batch
    for fs2, n, seed, fp in ((16000, 24000, 81, 5.0), (48000, 48000, 82, 1.0), (8000, 12000, 83, 10.0), (22050, 22050, 84, 2.5)):
        xs = synth_batch([seed], fs2, n).numpy()[0]
        po = port.harvest_option(); po.frame_period = fp
        ro = ref.harvest_option(); ro.frame_period = fp
        tp, fp_ = port.harvest(xs, fs2, po)
        tr, fr = ref.harvest(xs, fs2, ro)
        assert np.array_equal(tp, tr)
        assert not ((fp_ > 0) != (fr > 0)).any()
        assert rel_err(fp_, fr).max() < 1e-9, (fs2, fp)
        assert (fr > 0).sum() > 50


def test_port_synthesis_matches_reference(port, ref, golden):
    """Row f1: restated Synthesis (own FFTs, transform conventions written out) against the reference."""
    x, fs = pc.wav_from_golden(golden)
    fft = int(golden["fft_size"])
    sp = np.ascontiguousarray(golden["sp"]); ap = np.ascontiguousarray(golden["ap"])
    for key, fp, n in (("f0_stonemask", 5.0, len(x)), ("f0_dio_floor40", 5.0, len(x) + 3000), ("f0_stonemask", 4.0, len(x) // 2)):
        f0 = np.ascontiguousarray(golden[key])
        yp = port.synthesis(f0, sp, ap, fft, fp, fs, n)
        yr = ref.synthesis(f0, sp, ap, fft, fp, fs, n)
        assert np.abs(yr).max() > 0.1
        assert np.abs(yp - yr).max() <= 1e-12 * np.abs(yr).max()
