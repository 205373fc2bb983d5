"""CPU-side logic checks: the kernel sources compiled as a single-thread host emulation
(tests/emu) against the golden vectors and the compiled reference.  This is not the product
path (that is tests/test_gpu_parity.py, -m gpu); it exists so that arithmetic mistakes are caught
in the GPU-less build container."""
import os
import subprocess

import numpy as np
import pytest

import test_parity_common as pc


def test_reference_reproduces_its_own_goldens(ref, golden):
    """Only exercises the compiled reference when its results are recorded (WB_REF_RECORD, tests/refreplay.py): then
    it checks that the reference still gives the stored vaiueo2d vectors.  Replayed, it checks that the two stored
    sets agree."""
    x, fs = pc.wav_from_golden(golden)
    t, f0 = ref.dio(x, fs)
    assert np.array_equal(t, golden["time_axis"]) and np.array_equal(f0, golden["f0_dio"])
    f0 = ref.stonemask(x, fs, t, f0)
    assert np.array_equal(f0, golden["f0_stonemask"])
    assert np.ma.allequal(ref.cheaptrick(x, fs, t, f0), golden["sp"])
    assert np.ma.allequal(ref.d4c(x, fs, t, f0, int(golden["fft_size"])), golden["ap"])


def test_emu_randn_stream(emu, golden):
    pc.check_randn(emu, golden)


def test_emu_golden_cheaptrick_d4c_stonemask(emu, golden):
    pc.check_golden_cheaptrick_d4c_stonemask(emu, golden)


@pytest.mark.parametrize("fs,n,seeds", [(16000, 8000, [1, 2, 3]), (48000, 12000, [4]), (8000, 6000, [5])])
def test_emu_spectral_stages_on_reference_f0(emu, ref, fs, n, seeds):
    if fs == 8000:
        pytest.skip("fs < 15.8 kHz: D4C LoveTrain reads uninitialised memory in the reference (b2 > fft/2)")
    pc.check_batch_vs_ref(emu, ref, fs, n, seeds, f0_method="ref", ragged=len(seeds) > 1, stages=("sp", "ap"))


def test_emu_zero_tail(emu, ref):
    pc.check_batch_vs_ref(emu, ref, 16000, 8000, [7], f0_method="ref", zero_tail=3000, stages=("sp", "ap"))


def test_emu_golden_dio(emu, golden):
    pc.check_golden_dio(emu, golden)


@pytest.mark.parametrize("fs,n,seeds", [(16000, 16000, [11, 12, 13]), (48000, 14400, [14])])
def test_emu_dio_path_end_to_end(emu, ref, fs, n, seeds):
    pc.check_batch_vs_ref(emu, ref, fs, n, seeds, f0_method="dio", ragged=len(seeds) > 1)


def test_emu_dio_decimated(emu, ref):
    from synth import synth_batch
    x = synth_batch([21], 44100, 22050).numpy()
    o = emu.dio_option(); o.speed = 11
    ro = ref.dio_option(); ro.speed = 11
    t, f0, fl = emu.dio(x, 44100, o)
    emu.synchronize()
    tr, fr = ref.dio(x[0], 44100, ro)
    assert np.array_equal(t[0], tr)
    pc.assert_close(f0[0], fr, "DIO speed=11")


def test_emu_golden_harvest(emu, golden):
    pc.check_golden_harvest(emu, golden)


@pytest.mark.parametrize("fs,n,seeds", [(16000, 12000, [31, 32]), (48000, 9600, [33])])
def test_emu_harvest_path_end_to_end(emu, ref, fs, n, seeds):
    pc.check_batch_vs_ref(emu, ref, fs, n, seeds, f0_method="harvest", ragged=len(seeds) > 1)


def test_emu_harvest_frame_period_1ms(emu, ref):
    from synth import synth_batch
    x = synth_batch([41], 16000, 8000).numpy()
    o = emu.harvest_option(); o.frame_period = 1.0
    ro = ref.harvest_option(); ro.frame_period = 1.0
    t, f0, fl = emu.harvest(x, 16000, o)
    emu.synchronize()
    tr, fr = ref.harvest(x[0], 16000, ro)
    assert np.array_equal(t[0], tr)
    pc.assert_close(f0[0], fr, "Harvest 1 ms")


def test_emu_edge_cases(emu, ref):
    pc.check_edge_cases(emu, ref)


def test_emu_synthesis(emu, ref, golden):
    pc.check_synthesis(emu, ref, golden)


def test_emu_fft_known_answers(emu):
    pc.check_fft_known_answers(emu)


def test_emu_codec(emu, ref, golden):
    pc.check_codec(emu, ref, golden)


def test_emu_coded_frame_kernels(emu, ref, golden):
    pc.check_coded_frame_kernels(emu, ref, golden)


def test_emu_ingest(emu, ref, golden, tmp_path):
    pc.check_ingest(emu, golden, ref, tmp_path)


def test_emu_analyze_coded_host(emu, golden):
    pc.check_analyze_coded(emu, golden)


def test_emu_analyze_batch(emu, golden):
    pc.check_analyze_batch(emu, golden)


def test_emu_host_pipeline_chunking(emu, golden):
    pc.check_host_pipeline_chunking(emu, golden)


def test_emu_dio_agrees_with_port(emu):
    """Two independent time-domain implementations of Dio (the kernel sources and oracle/world_oracle.cpp), both
    with the ripple of the reference's spectral mirroring loop written out, agree to rounding."""
    from refworld import RefWorld, ORACLE_LIB, rel_err
    from synth import synth_batch
    subprocess.check_call(["make", "-s", "-C", os.path.join(pc.os.path.dirname(pc.os.path.dirname(pc.os.path.abspath(pc.__file__))), "oracle"),
                           "libworld_oracle.so"])
    port = RefWorld(ORACLE_LIB)
    for fs, n, seed, speed in ((16000, 16000, 71, 1), (44100, 22050, 72, 11), (48000, 24000, 73, 4)):
        x = synth_batch([seed], fs, n).numpy()
        po = port.dio_option(); po.speed = speed
        eo = emu.dio_option(); eo.speed = speed
        tp, fp = port.dio(x[0], fs, po)
        te, fe, fl = emu.dio(x, fs, eo)
        emu.synchronize()
        assert np.array_equal(te[0], tp)
        assert rel_err(fe[0], fp).max() < 1e-12


def test_emu_event_dense_and_degenerate_bands(emu, ref):
    pc.check_event_dense_and_degenerate_bands(emu, ref)


def test_emu_zero_tail_f0(emu, ref):
    pc.check_zero_tail_f0(emu, ref)


def test_emu_harvest_per_frame_refinement(emu, ref):
    """The per-frame refinement kernel (WB_NO_REFINE_CHAIN=1): the default since round 2 is the chain kernel
    (one template per base candidate shared by its seven overlapped frames) wherever a 1 ms frame is a whole
    number of decimated samples; the per-frame kernel still serves the other rates (22.05 / 44.1 kHz) and must
    give the same contour everywhere.  Same tolerance, no V/UV flip."""
    from refworld import rel_err
    from synth import synth_batch
    saved = os.environ.get("WB_NO_REFINE_CHAIN")
    os.environ["WB_NO_REFINE_CHAIN"] = "1"
    try:
        for fs, n, seeds, fp in ((16000, 16000, [1, 2], 5.0), (48000, 24000, [3], 1.0), (8000, 8000, [6], 2.5)):
            x = synth_batch(seeds, fs, n).numpy()
            lens = [n - 1234 * u for u in range(len(seeds))]
            o = emu.harvest_option(); o.frame_period = fp
            ro = ref.harvest_option(); ro.frame_period = fp
            t, f, fl = emu.harvest(x, fs, o, x_lengths=lens)
            emu.synchronize()
            for u in range(len(seeds)):
                tr, fr = ref.harvest(x[u, :lens[u]], fs, ro)
                got = f[u, :fl[u]]
                assert np.array_equal(t[u, :fl[u]], tr)
                assert not ((got > 0) != (fr > 0)).any()
                assert rel_err(got, fr).max() <= pc.TOL
                assert (fr > 0).sum() > 50
    finally:
        if saved is None:
            os.environ.pop("WB_NO_REFINE_CHAIN", None)
        else:
            os.environ["WB_NO_REFINE_CHAIN"] = saved


def test_emu_dio_silence_onset_is_bounded(emu, ref):
    pc.check_dio_silence_onset_bound(emu, ref)


def test_emu_mirroring_ripple_cases(emu, ref):
    pc.check_mirroring_ripple_cases(emu, ref)


def test_emu_argument_errors(emu):
    """The batched ABI answers bad arguments with an error code and a message instead of the reference's undefined
    behaviour; empty batches are fine."""
    import ctypes as C
    from world_b200 import api
    lib, h = emu.lib, emu._h
    fs = 16000
    x = np.zeros((2, 800)); t = np.zeros((2, 11)); f0 = np.zeros((2, 11)); sp = np.zeros((2, 11, 513))
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    do = emu.dio_option(); ho = emu.harvest_option(); co = emu.cheaptrick_option(fs); d4 = emu.d4c_option()
    ok, einval = 0, 3
    # empty batch
    assert lib.world_b200_dio_batch(h, P(x), 0, 800, None, fs, C.byref(do), P(t), P(f0), 11) == ok
    assert lib.world_b200_harvest_batch(h, P(x), 0, 800, None, fs, C.byref(ho), P(t), P(f0), 11) == ok
    # null pointers, negative counts, bad rates
    assert lib.world_b200_dio_batch(h, None, 2, 800, None, fs, C.byref(do), P(t), P(f0), 11) == einval
    assert lib.world_b200_dio_batch(h, P(x), -1, 800, None, fs, C.byref(do), P(t), P(f0), 11) == einval
    assert lib.world_b200_harvest_batch(h, P(x), 2, 800, None, 0, C.byref(ho), P(t), P(f0), 11) == einval
    # rows shorter than the frame count / lengths beyond the row
    assert lib.world_b200_dio_batch(h, P(x), 2, 800, None, fs, C.byref(do), P(t), P(f0), 5) == einval
    assert b"f0_stride" in lib.world_b200_last_error(h)
    lens = (C.c_int * 2)(800, 801)
    assert lib.world_b200_cheaptrick_batch(h, P(x), 2, 800, lens, fs, P(t), P(f0), None, 11, C.byref(co), P(sp)) == einval
    # fft sizes the on-chip transforms cannot do
    bad = api.CheapTrickOption(); bad.q1 = -0.15; bad.f0_floor = 71.0; bad.fft_size = 1000
    assert lib.world_b200_cheaptrick_batch(h, P(x), 2, 800, None, fs, P(t), P(f0), None, 11, C.byref(bad), P(sp)) == einval
    # (D4C's fft_size only sets the width of the output rows, fft_size / 2 + 1: any value is legal, as in the reference)
    assert lib.world_b200_d4c_batch(h, P(x), 2, 800, None, fs, P(t), P(f0), None, 11, 1000, C.byref(d4), P(sp)) == ok
    assert lib.world_b200_code_spectral_envelope_batch(h, P(sp), 2, None, 11, fs, 1000, 40, P(sp)) == einval
    assert lib.world_b200_code_spectral_envelope_batch(h, P(sp), 2, None, 11, fs, 1024, 400, P(sp)) == einval
    assert lib.world_b200_pcm_to_double_batch(h, P(x), 12, 2, 800, None, P(x)) == einval
    assert lib.world_b200_synthesis_batch(h, P(f0), None, 2, 11, P(sp), P(sp), 1000, 5.0, fs, None, 800, P(x)) == einval
    emu.synchronize()      # none of the rejected calls left the context in an error state
