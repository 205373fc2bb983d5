"""Parity tests proper: the CUDA library (through the C ABI) against the golden vectors and the
compiled reference, on a real B200.  Tolerance 1e-6 relative (north_star); integers bit exact."""
import numpy as np
import pytest

import test_parity_common as pc

pytestmark = pytest.mark.gpu


def test_gpu_randn_stream(gpu_world, golden):
    pc.check_randn(gpu_world, golden)


def test_gpu_golden_cheaptrick_d4c_stonemask(gpu_world, golden):
    pc.check_golden_cheaptrick_d4c_stonemask(gpu_world, golden)


@pytest.mark.parametrize("fs,n,seeds", [(16000, 16000, [1, 2, 3, 4, 5]), (48000, 24000, [6, 7]), (22050, 11025, [8])])
def test_gpu_spectral_stages_on_reference_f0(gpu_world, ref, fs, n, seeds):
    pc.check_batch_vs_ref(gpu_world, ref, fs, n, seeds, f0_method="ref", ragged=len(seeds) > 1, stages=("sp", "ap"))


def test_gpu_zero_tail(gpu_world, ref):
    pc.check_batch_vs_ref(gpu_world, ref, 16000, 16000, [9], f0_method="ref", zero_tail=6000, stages=("sp", "ap"))


def test_gpu_golden_dio(gpu_world, golden):
    pc.check_golden_dio(gpu_world, golden)


@pytest.mark.parametrize("fs,n,seeds", [(16000, 48000, [11, 12, 13, 14]), (48000, 48000, [15, 16]), (22050, 22050, [17])])
def test_gpu_dio_path_end_to_end(gpu_world, ref, fs, n, seeds):
    pc.check_batch_vs_ref(gpu_world, ref, fs, n, seeds, f0_method="dio", ragged=len(seeds) > 1)


def test_gpu_dio_decimated(gpu_world, ref):
    import torch
    from synth import synth_batch
    x = synth_batch([21], 44100, 44100)
    o = gpu_world.dio_option(); o.speed = 11
    ro = ref.dio_option(); ro.speed = 11
    t, f0, fl = gpu_world.dio(x.cuda(), 44100, o)
    gpu_world.synchronize()
    tr, fr = ref.dio(x[0].numpy(), 44100, ro)
    assert np.array_equal(t[0].cpu().numpy(), tr)
    pc.assert_close(f0[0], fr, "DIO speed=11")


def test_gpu_golden_harvest(gpu_world, golden):
    pc.check_golden_harvest(gpu_world, golden)


@pytest.mark.parametrize("fs,n,seeds", [(16000, 48000, [31, 32, 33, 34]), (48000, 48000, [35, 36]), (22050, 22050, [37])])
def test_gpu_harvest_path_end_to_end(gpu_world, ref, fs, n, seeds):
    pc.check_batch_vs_ref(gpu_world, ref, fs, n, seeds, f0_method="harvest", ragged=len(seeds) > 1)


def test_gpu_edge_cases(gpu_world, ref):
    pc.check_edge_cases(gpu_world, ref)


def test_gpu_long_48k_utterance(gpu_world, ref):
    """BASELINE configs[3] shape: 48 kHz, CheapTrick fft 2048 + D4C fft 4096 (long-FFT shared-memory path)."""
    import torch
    from synth import synth_batch
    fs, n = 48000, 48000 * 6
    x = synth_batch([71], fs, n)
    xh = x[0].numpy()
    tr, fr = ref.dio(xh, fs)
    fr = ref.stonemask(xh, fs, tr, fr)
    xb = x.cuda()
    t, f0, fl = gpu_world.dio(xb, fs)
    f0 = gpu_world.stonemask(xb, fs, t, f0)
    opt = gpu_world.cheaptrick_option(fs)
    assert opt.fft_size == 2048
    sp = gpu_world.cheaptrick(xb, fs, t, f0, opt)
    ap = gpu_world.d4c(xb, fs, t, f0, opt.fft_size)
    gpu_world.synchronize()
    assert np.array_equal(t[0].cpu().numpy(), tr)
    pc.assert_close(f0[0], fr, "f0 48k")
    fu = np.ascontiguousarray(f0[0].cpu().numpy())
    pc.assert_close(sp[0], ref.cheaptrick(xh, fs, tr, fu, opt), "sp 48k")
    pc.assert_close(ap[0], ref.d4c(xh, fs, tr, fu, opt.fft_size), "ap 48k")


def test_gpu_legacy_api_and_analyze_host(gpu_world, ref, golden):
    """The reference's own entry points (host pointers, double**) and the one-call host pipeline."""
    import ctypes as C
    from world_b200 import api
    lib = gpu_world.lib
    x, fs = pc.wav_from_golden(golden)
    n = len(x)
    L = lib.GetSamplesForDIO(fs, n, 5.0)
    t = np.zeros(L); f0 = np.zeros(L); f0r = np.zeros(L)
    do = api.DioOption(); lib.InitializeDioOption(C.byref(do))
    lib.Dio(x.ctypes.data, n, fs, C.byref(do), t.ctypes.data, f0.ctypes.data)
    lib.StoneMask(x.ctypes.data, n, fs, t.ctypes.data, f0.ctypes.data, L, f0r.ctypes.data)
    co = api.CheapTrickOption(); lib.InitializeCheapTrickOption(fs, C.byref(co))
    bins = co.fft_size // 2 + 1
    sp = np.zeros((L, bins)); ap = np.zeros((L, bins))
    rows = (C.c_void_p * L)(*[sp[i].ctypes.data for i in range(L)])
    lib.CheapTrick(x.ctypes.data, n, fs, t.ctypes.data, f0r.ctypes.data, L, C.byref(co), rows)
    rows2 = (C.c_void_p * L)(*[ap[i].ctypes.data for i in range(L)])
    d4 = api.D4COption(); lib.InitializeD4COption(C.byref(d4))
    lib.D4C(x.ctypes.data, n, fs, t.ctypes.data, f0r.ctypes.data, L, co.fft_size, C.byref(d4), rows2)
    assert np.array_equal(t, golden["time_axis"])
    pc.assert_close(f0, golden["f0_dio"], "legacy Dio")
    pc.assert_close(f0r, golden["f0_stonemask"], "legacy StoneMask")
    pc.assert_close(sp, ref.cheaptrick(x, fs, t, f0r), "legacy CheapTrick")
    pc.assert_close(ap, ref.d4c(x, fs, t, f0r, co.fft_size), "legacy D4C")
    fh = np.zeros(L); th = np.zeros(L)
    ho = api.HarvestOption(); lib.InitializeHarvestOption(C.byref(ho))
    lib.Harvest(x.ctypes.data, n, fs, C.byref(ho), th.ctypes.data, fh.ctypes.data)
    pc.assert_close(fh, golden["f0_harvest"], "legacy Harvest")
    # one-call host pipeline on a small batch (both F0 methods)
    xb = np.ascontiguousarray(np.stack([x, x[::-1]]))
    for method, key in ((api.F0_DIO_STONEMASK, "f0_stonemask"), (api.F0_HARVEST, "f0_harvest")):
        ao = gpu_world.analysis_option(fs, method)
        ta, fa, spa, apa, fl = gpu_world.analyze_host(xb, fs, ao)
        assert np.array_equal(ta[0], golden["time_axis"])
        pc.assert_close(fa[0], golden[key], "analyze_host f0")
        pc.assert_close(spa[0], ref.cheaptrick(x, fs, ta[0], np.ascontiguousarray(fa[0])), "analyze_host sp")
        pc.assert_close(apa[0], ref.d4c(x, fs, ta[0], np.ascontiguousarray(fa[0]), co.fft_size), "analyze_host ap")


def test_gpu_synthesis(gpu_world, ref, golden):
    pc.check_synthesis(gpu_world, ref, golden)


def test_gpu_legacy_synthesis(gpu_world, ref, golden):
    import ctypes as C
    x, fs = pc.wav_from_golden(golden)
    # the reference's own CheapTrick / D4C rows of the DIO path (the stored vectors) as the parameters
    f0 = np.ascontiguousarray(golden["f0_stonemask"])
    sp = np.ascontiguousarray(golden["sp"]); ap = np.ascontiguousarray(golden["ap"])
    y = np.zeros(len(x))
    rows_s = (C.c_void_p * len(f0))(*[sp[i].ctypes.data for i in range(len(f0))])
    rows_a = (C.c_void_p * len(f0))(*[ap[i].ctypes.data for i in range(len(f0))])
    gpu_world.lib.Synthesis(f0.ctypes.data, len(f0), rows_s, rows_a, 1024, 5.0, fs, len(x), y.ctypes.data)
    yr = ref.synthesis(f0, sp, ap, 1024, 5.0, fs, len(x))
    assert np.abs(y - yr).max() <= 1e-9 * np.abs(yr).max()


def test_gpu_fft_known_answers(gpu_world):
    pc.check_fft_known_answers(gpu_world)


def test_gpu_codec(gpu_world, ref, golden):
    pc.check_codec(gpu_world, ref, golden)


def test_gpu_coded_frame_kernels(gpu_world, ref, golden):
    pc.check_coded_frame_kernels(gpu_world, ref, golden)


def test_gpu_ingest(gpu_world, ref, golden, tmp_path):
    pc.check_ingest(gpu_world, golden, ref, tmp_path)


def test_gpu_analyze_coded_host(gpu_world, golden):
    from world_b200 import api
    pc.check_analyze_coded(gpu_world, golden, api.F0_DIO_STONEMASK)


def test_gpu_legacy_codec(gpu_world, ref, golden):
    """codec.h entry points with the reference's calling convention (row pointers, host memory)."""
    import ctypes as C
    lib = gpu_world.lib
    fs, fft, dims = int(golden["fs"]), int(golden["fft_size"]), int(golden["coded_dims"])
    sp = np.ascontiguousarray(golden["sp"]); ap = np.ascontiguousarray(golden["ap"])
    L = sp.shape[0]
    rows = lambda a: (C.c_void_p * a.shape[0])(*[a[i].ctypes.data for i in range(a.shape[0])])
    n_ap = lib.GetNumberOfAperiodicities(fs)
    assert n_ap == ref.number_of_aperiodicities(fs)
    csp = np.zeros((L, dims)); cap = np.zeros((L, n_ap)); dsp = np.zeros_like(sp); dap = np.zeros_like(ap)
    lib.CodeSpectralEnvelope(rows(sp), L, fs, fft, dims, rows(csp))
    lib.CodeAperiodicity(rows(ap), L, fs, fft, rows(cap))
    lib.DecodeSpectralEnvelope(rows(csp), L, fs, fft, dims, rows(dsp))
    lib.DecodeAperiodicity(rows(cap), L, fs, fft, rows(dap))
    pc.assert_close_signed(csp, golden["coded_sp"], "legacy CodeSpectralEnvelope")
    pc.assert_close_signed(cap, golden["coded_ap"], "legacy CodeAperiodicity")
    pc.assert_close(dsp[::4], golden["decoded_sp_rows"], "legacy DecodeSpectralEnvelope")
    pc.assert_close(dap[::4], golden["decoded_ap_rows"], "legacy DecodeAperiodicity")


def test_gpu_dio_silence_onset_is_bounded(gpu_world, ref):
    pc.check_dio_silence_onset_bound(gpu_world, ref)


def test_gpu_analyze_batch_lanes(gpu_world, golden):
    pc.check_analyze_batch(gpu_world, golden)


def test_gpu_host_pipeline_chunking(gpu_world, golden):
    from world_b200 import api
    pc.check_host_pipeline_chunking(gpu_world, golden, api.F0_DIO_STONEMASK)
    pc.check_host_pipeline_chunking(gpu_world, golden, api.F0_HARVEST)


def test_gpu_event_dense_and_degenerate_bands(gpu_world, ref):
    pc.check_event_dense_and_degenerate_bands(gpu_world, ref)


def test_gpu_zero_tail_f0(gpu_world, ref):
    pc.check_zero_tail_f0(gpu_world, ref)


def test_gpu_mirroring_ripple_cases(gpu_world, ref):
    pc.check_mirroring_ripple_cases(gpu_world, ref)


def test_gpu_benchmark_scale_batch(gpu_world, ref):
    """Parity at the scale the headline number is quoted on: 600 utterances x 10 s @16 kHz through the one-call
    device path (world_b200_analyze_batch: two utterance slices on two streams, Harvest in its real passes with the
    edge-list / candidate capacities of 10 s utterances), then the reference's own chain -- its Harvest f0 feeding
    its CheapTrick and D4C -- on eight utterances including the first and last rows of every slice."""
    import torch
    from synth import synth_batch
    from world_b200 import api
    fs, n, U = 16000, 160000, 600
    dev = f"cuda:{gpu_world.device}"
    x = torch.empty((U, n), dtype=torch.float64, device=dev)
    for u0 in range(0, U, 50):
        x[u0:u0 + 50] = synth_batch(range(7001 + u0, 7051 + u0), fs, n, device=dev)
    opt = gpu_world.analysis_option(fs, api.F0_HARVEST)
    t, f0, sp, ap, fl = gpu_world.analyze_batch(x, fs, opt)
    gpu_world.synchronize()
    assert fl == [2001] * U
    flips = frames = 0
    worst = {"f0": 0.0, "sp": 0.0, "ap": 0.0}
    for u in (0, 1, 150, 299, 300, 301, 450, 599):
        xu = x[u].cpu().numpy()
        tr, fr = ref.harvest(xu, fs)
        o = ref.cheaptrick_option(fs)
        spr = ref.cheaptrick(xu, fs, tr, fr, o)
        apr = ref.d4c(xu, fs, tr, fr, o.fft_size)
        g = f0[u].cpu().numpy()
        assert np.array_equal(t[u].cpu().numpy(), tr)
        flips += int(((g > 0) != (fr > 0)).sum())
        frames += len(fr)
        worst["f0"] = max(worst["f0"], pc.rel_err(g, fr).max())
        worst["sp"] = max(worst["sp"], pc.rel_err(sp[u].cpu().numpy(), spr).max())
        worst["ap"] = max(worst["ap"], pc.rel_err(ap[u].cpu().numpy(), apr).max())
        assert (fr > 0).sum() > 1000
    assert flips == 0, f"{flips} V/UV flips in {frames} frames"
    assert max(worst.values()) <= pc.TOL, worst


def test_gpu_unsupported_configurations_fail_cleanly(gpu_world):
    """Where the on-chip tables / shared memory end (DESIGN.md, INTEGRATION.md 4) the library returns
    WORLD_B200_EINVAL with a message -- no kernel fault, no sticky CUDA error, and the context keeps working."""
    import torch
    from world_b200.api import WorldError
    from synth import synth_batch
    dev = f"cuda:{gpu_world.device}"
    w = gpu_world
    cases = []
    # StoneMask / D4C above the twiddle table: fs = 192 kHz
    x = torch.zeros((1, 19200), dtype=torch.float64, device=dev)
    t = torch.arange(21, dtype=torch.float64, device=dev)[None] * 0.005
    f = torch.full((1, 21), 150.0, dtype=torch.float64, device=dev)
    cases.append(("StoneMask fs=192k", lambda: w.stonemask(x, 192000, t, f)))
    cases.append(("D4C fs=192k", lambda: w.d4c(x, 192000, t, f, 8192)))
    # Harvest with a floor whose refinement window / band filters do not fit on chip
    o = w.harvest_option(); o.f0_floor = 8.0
    cases.append(("Harvest floor 8 Hz", lambda: w.harvest(x[:, :16000], 16000, o)))
    # DIO at 48 kHz, speed 1, very low floor: low-pass windows of thousands of taps
    do = w.dio_option(); do.f0_floor = 5.0
    cases.append(("Dio floor 5 Hz @48k", lambda: w.dio(x, 48000, do)))
    # CheapTrick with a non power-of-two fft_size
    co = w.cheaptrick_option(16000); co.fft_size = 1000
    cases.append(("CheapTrick fft 1000", lambda: w.cheaptrick(x[:, :16000], 16000, t, f, co)))
    for name, call in cases:
        with pytest.raises(WorldError, match="error 3"):
            call()
    # ... and the context is still healthy
    xs = synth_batch([3], 16000, 8000, device=dev)
    tt, ff, fl = w.harvest(xs, 16000)
    w.synchronize()
    assert (ff > 0).any()
