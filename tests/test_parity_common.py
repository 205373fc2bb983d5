"""Shared parity checks; the same assertions run against the host emulation (CPU, -m "not gpu")
and against the CUDA library (-m gpu).  Tolerance: BASELINE.json's north_star -- 1e-6 relative
for f0 / spectrogram / aperiodicity, frame counts and time_axis bit-exact."""
import os

import numpy as np

from refworld import rel_err

TOL = 1e-6


def to_np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def make(world, a, dtype=np.float64):
    """host array -> the array type `world` works on"""
    a = np.ascontiguousarray(a, dtype=dtype)
    if world.xp == "torch":
        import torch
        return torch.from_numpy(a).to(f"cuda:{world.device}")
    return a


def wav_from_golden(golden):
    return golden["pcm"].astype(np.float64) / 32768.0, int(golden["fs"])


def assert_close(got, want, what, tol=TOL):
    r = rel_err(to_np(got), want)
    assert r.max() <= tol, f"{what}: max rel err {r.max():.3e}, {(r > tol).mean():.2%} of entries beyond {tol}"


def check_randn(world, golden):
    n = 1000008
    out = make(world, np.zeros(n, dtype=np.uint32), dtype=np.uint32)
    world.randn_stream(n, out)
    world.synchronize()
    vals = to_np(out).astype(np.float64) / 268435456.0 - 6.0
    assert np.array_equal(vals[:32], golden["randn_first32"])      # bit exact
    assert np.array_equal(vals[1000000:1000008], golden["randn_at_1e6"])


def check_golden_cheaptrick_d4c_stonemask(world, golden):
    x, fs = wav_from_golden(golden)
    xb = make(world, x[None, :])
    t = make(world, golden["time_axis"][None, :])
    f0 = make(world, golden["f0_stonemask"][None, :])
    fft = int(golden["fft_size"])
    opt = world.cheaptrick_option(fs)
    assert opt.fft_size == fft
    sp = world.cheaptrick(xb, fs, t, f0, opt)
    ap = world.d4c(xb, fs, t, f0, fft)
    sm = world.stonemask(xb, fs, t, make(world, golden["f0_dio"][None, :]))
    sm40 = world.stonemask(xb, fs, t, make(world, golden["f0_dio_floor40"][None, :]))
    world.synchronize()
    assert_close(sp[0], golden["sp"], "spectrogram (vaiueo2d, DIO path)")
    assert_close(ap[0], golden["ap"], "aperiodicity (vaiueo2d, DIO path)")
    assert_close(sm[0], golden["f0_stonemask"], "StoneMask f0")
    assert_close(sm40[0], golden["f0_stonemask_floor40"], "StoneMask f0 (floor 40)")
    # Harvest-path f0 through the same kernels (rows subsampled in the fixture)
    f0h = make(world, golden["f0_harvest"][None, :])
    sp_h = world.cheaptrick(xb, fs, t, f0h, opt)
    ap_h = world.d4c(xb, fs, t, f0h, fft)
    world.synchronize()
    assert_close(to_np(sp_h)[0][::4], golden["sp_harvest_rows"], "spectrogram (Harvest f0)")
    assert_close(to_np(ap_h)[0][::4], golden["ap_harvest_rows"], "aperiodicity (Harvest f0)")


def check_batch_vs_ref(world, ref, fs, n_samples, seeds, f0_method="dio", zero_tail=0, ragged=False,
                       stages=("f0", "sp", "ap")):
    """Synthetic ragged batch through the batched ABI vs the reference run utterance by utterance."""
    from synth import synth_batch
    x = synth_batch(seeds, fs, n_samples, device="cpu", zero_tail=zero_tail).numpy()
    n = len(seeds)
    lens = [n_samples - (37 * i * (fs // 100)) % (n_samples // 3) for i in range(n)] if ragged else [n_samples] * n
    xb = make(world, x)
    if f0_method == "dio":
        t, f0, fl = world.dio(xb, fs, x_lengths=lens)
        f0 = world.stonemask(xb, fs, t, f0, x_lengths=lens, f0_lengths=fl)
    elif f0_method == "harvest":
        t, f0, fl = world.harvest(xb, fs, x_lengths=lens)
    else:  # reference f0 handed in
        fl = [ref.frames(fs, l) for l in lens]
        tn = np.zeros((n, max(fl))); fn = np.zeros((n, max(fl)))
        for u in range(n):
            tr, fr = ref.dio(x[u, :lens[u]], fs)
            fn[u, :fl[u]] = ref.stonemask(x[u, :lens[u]], fs, tr, fr); tn[u, :fl[u]] = tr
        t, f0 = make(world, tn), make(world, fn)
    opt = world.cheaptrick_option(fs)
    sp = world.cheaptrick(xb, fs, t, f0, opt, x_lengths=lens, f0_lengths=fl) if "sp" in stages else None
    ap = world.d4c(xb, fs, t, f0, opt.fft_size, x_lengths=lens, f0_lengths=fl) if "ap" in stages else None
    world.synchronize()
    t, f0 = to_np(t), to_np(f0)
    flips = 0
    for u in range(n):
        xu = x[u, :lens[u]]
        if f0_method == "harvest":
            tr, fr = ref.harvest(xu, fs)
        else:
            tr, fr = ref.dio(xu, fs)
            fr = ref.stonemask(xu, fs, tr, fr)
        assert len(tr) == fl[u]
        assert np.array_equal(t[u, :fl[u]], tr), "time_axis must be bit exact"
        if "f0" in stages:
            flips += int(np.sum((f0[u, :fl[u]] == 0) != (fr == 0)))
            assert_close(f0[u, :fl[u]], fr, f"f0 utt {u}")
        # spectral stages are compared on the f0 the GPU path produced (== reference within 1e-6,
        # but window lengths derive from it, so hand the reference exactly the same values)
        fu = np.ascontiguousarray(f0[u, :fl[u]])
        if sp is not None:
            assert_close(to_np(sp)[u, :fl[u]], ref.cheaptrick(xu, fs, tr, fu, opt), f"spectrogram utt {u}")
        if ap is not None:
            assert_close(to_np(ap)[u, :fl[u]], ref.d4c(xu, fs, tr, fu, opt.fft_size), f"aperiodicity utt {u}")
    assert flips == 0


def check_golden_dio(world, golden):
    x, fs = wav_from_golden(golden)
    xb = make(world, x[None, :])
    t, f0, fl = world.dio(xb, fs)
    o = world.dio_option(); o.f0_floor = 40.0
    _, f0_40, _ = world.dio(xb, fs, o)
    world.synchronize()
    assert fl[0] == len(golden["time_axis"])
    assert np.array_equal(to_np(t)[0], golden["time_axis"])
    assert_close(f0[0], golden["f0_dio"], "DIO f0")
    assert_close(f0_40[0], golden["f0_dio_floor40"], "DIO f0 (floor 40)")


def check_golden_harvest(world, golden):
    x, fs = wav_from_golden(golden)
    xb = make(world, x[None, :])
    t, f0, fl = world.harvest(xb, fs)
    o = world.harvest_option(); o.f0_floor = 40.0
    _, f0_40, _ = world.harvest(xb, fs, o)
    world.synchronize()
    assert np.array_equal(to_np(t)[0], golden["time_axis"])
    assert_close(f0[0], golden["f0_harvest"], "Harvest f0")
    assert_close(f0_40[0], golden["f0_harvest_floor40"], "Harvest f0 (floor 40)")


def check_edge_cases(world, ref):
    """Silence, very short and ragged utterances, non-default frame periods."""
    from synth import synth_batch
    fs = 16000
    x = synth_batch([61, 62, 63], fs, 8000).numpy()
    x[1, :] = 0.0                      # digital silence: f0 = 0 everywhere, randn-only frames downstream
    lens = [8000, 8000, 900]           # third utterance is shorter than most analysis windows
    xb = make(world, x)
    for method in ("dio", "harvest"):
        for fp in (5.0, 10.0, 2.5):
            if method == "dio":
                o = world.dio_option(); o.frame_period = fp
                ro = ref.dio_option(); ro.frame_period = fp
                t, f0, fl = world.dio(xb, fs, o, x_lengths=lens)
            else:
                o = world.harvest_option(); o.frame_period = fp
                ro = ref.harvest_option(); ro.frame_period = fp
                t, f0, fl = world.harvest(xb, fs, o, x_lengths=lens)
            world.synchronize()
            for u in range(3):
                xu = x[u, :lens[u]]
                tr, fr = (ref.dio(xu, fs, ro) if method == "dio" else ref.harvest(xu, fs, ro))
                assert fl[u] == len(tr)
                assert np.array_equal(to_np(t)[u, :fl[u]], tr)
                assert_close(to_np(f0)[u, :fl[u]], fr, f"{method} fp={fp} utt {u}")
    # spectral stages on the silent and the short utterance (reference f0)
    fl = [ref.frames(fs, l) for l in lens]
    tn = np.zeros((3, max(fl))); fn = np.zeros((3, max(fl)))
    for u in range(3):
        tr, fr = ref.dio(x[u, :lens[u]], fs)
        tn[u, :fl[u]] = tr; fn[u, :fl[u]] = ref.stonemask(x[u, :lens[u]], fs, tr, fr)
    t, f0 = make(world, tn), make(world, fn)
    opt = world.cheaptrick_option(fs)
    sp = world.cheaptrick(xb, fs, t, f0, opt, x_lengths=lens, f0_lengths=fl)
    ap = world.d4c(xb, fs, t, f0, opt.fft_size, x_lengths=lens, f0_lengths=fl)
    world.synchronize()
    for u in range(3):
        xu = x[u, :lens[u]]
        assert_close(to_np(sp)[u, :fl[u]], ref.cheaptrick(xu, fs, tn[u, :fl[u]], fn[u, :fl[u]], opt), f"sp edge utt {u}")
        assert_close(to_np(ap)[u, :fl[u]], ref.d4c(xu, fs, tn[u, :fl[u]], fn[u, :fl[u]], opt.fft_size), f"ap edge utt {u}")


def check_synthesis(world, ref, golden):
    """SURVEY.md 8 row f1: batched Synthesis() vs the reference (relative to the waveform peak)."""
    from synth import synth_batch
    x, fs = wav_from_golden(golden)
    fft = int(golden["fft_size"])
    f0 = golden["f0_stonemask"]; sp = golden["sp"]; ap = golden["ap"]
    yr = ref.synthesis(f0, sp, ap, fft, 5.0, fs, len(x))
    y = world.synthesis(make(world, f0[None]), make(world, sp[None]), make(world, ap[None]), fft, 5.0, fs, len(x))
    world.synchronize()
    assert np.abs(to_np(y)[0] - yr).max() <= 1e-9 * np.abs(yr).max()
    # ragged synthetic batch: the reference's f0, envelope and aperiodicity from this library on that f0; both
    # synthesizers get the same parameters
    fs2, n = 16000, 12000
    xs = synth_batch([81, 82], fs2, n).numpy()
    lens = [12000, 9000]
    L = [ref.frames(fs2, l) for l in lens]
    opt = ref.cheaptrick_option(fs2)
    bins = opt.fft_size // 2 + 1
    F = np.zeros((2, max(L))); S = np.ones((2, max(L), bins)); A = np.ones((2, max(L), bins))
    refs = []
    for u in range(2):
        xu = xs[u, :lens[u]]
        t, f = ref.harvest(xu, fs2)
        xw, tw, fw = make(world, xu[None]), make(world, t[None]), make(world, f[None])
        s_ = to_np(world.cheaptrick(xw, fs2, tw, fw, opt))[0]
        a_ = to_np(world.d4c(xw, fs2, tw, fw, opt.fft_size))[0]
        world.synchronize()
        F[u, :L[u]] = f; S[u, :L[u]] = s_; A[u, :L[u]] = a_
        refs.append(ref.synthesis(f, s_, a_, opt.fft_size, 5.0, fs2, lens[u]))
    y = world.synthesis(make(world, F), make(world, S), make(world, A), opt.fft_size, 5.0, fs2, n, f0_lengths=L,
                        y_lengths=lens)
    world.synchronize()
    for u in range(2):
        assert np.abs(to_np(y)[u, :lens[u]] - refs[u]).max() <= 1e-9 * np.abs(refs[u]).max(), f"synthesis utt {u}"


def check_fft_known_answers(world):
    """The shared-memory FFT against numpy's (conventions of SURVEY.md App. A0), every size it serves."""
    rng = np.random.RandomState(7)
    for lg in range(2, 14):
        n = 1 << lg
        x = rng.standard_normal(n)
        want = np.fft.rfft(x)
        for name in ("rfft_test", "sfft_test"):   # in-place DIT (synthesis, codec) / self-sorting padded (frame kernels)
            out = make(world, np.zeros(n + 2))
            getattr(world, name)(make(world, x), out)
            world.synchronize()
            got = to_np(out).reshape(-1, 2)
            err = np.abs(got[:, 0] + 1j * got[:, 1] - want).max() / np.abs(want).max()
            assert err < 1e-13, f"{name} n={n}: {err:.2e}"


# ---------------------------------------------------------------- codec (row f2) and ingest (row f3)
def assert_close_signed(got, want, what, tol=TOL):
    """Cepstral coefficients and dB values pass through zero, so the relative bound is taken against
    max(|want|, 1e-4 * max|want| of the whole array): 1e-6 of anything that is not numerically zero."""
    want = np.ma.asarray(want)
    r = rel_err(to_np(got), want, floor=1e-4 * np.abs(want).max())
    assert r.max() <= tol, f"{what}: max rel err {r.max():.3e}"


def check_codec(world, ref, golden):
    fs, fft, dims = int(golden["fs"]), int(golden["fft_size"]), int(golden["coded_dims"])
    sp, ap = make(world, golden["sp"][None]), make(world, golden["ap"][None])
    csp = world.code_spectral_envelope(sp, fs, fft, dims)
    cap = world.code_aperiodicity(ap, fs, fft)
    dsp = world.decode_spectral_envelope(make(world, golden["coded_sp"][None]), fs, fft, dims)
    dap = world.decode_aperiodicity(make(world, golden["coded_ap"][None]), fs, fft)
    world.synchronize()
    assert world.number_of_aperiodicities(fs) == golden["coded_ap"].shape[1]
    assert_close_signed(csp[0], golden["coded_sp"], "coded spectral envelope (golden)")
    assert_close_signed(cap[0], golden["coded_ap"], "coded aperiodicity (golden)")
    assert_close(to_np(dsp)[0][::4], golden["decoded_sp_rows"], "decoded spectral envelope (golden)")
    assert_close(to_np(dap)[0][::4], golden["decoded_ap_rows"], "decoded aperiodicity (golden)")
    # other rates / sizes / dimensions against the compiled reference, ragged batch of three
    for fs2, fft2 in [(16000, 1024), (48000, 2048), (8000, 512), (44100, 2048), (16000, 4096)]:
        rng = np.random.default_rng(fs2 + fft2)
        bins, lens = fft2 // 2 + 1, [9, 4, 0]
        sp2 = np.exp(rng.normal(size=(3, 9, bins)) * 3 - 8)
        ap2 = np.clip(rng.uniform(size=(3, 9, bins)), 1e-3, 1 - 1e-12)
        ap2[0, 2] = 1 - 1e-12                                   # an unvoiced frame (decodes to the constant)
        n_ap = ref.number_of_aperiodicities(fs2)
        assert world.number_of_aperiodicities(fs2) == n_ap
        for d in (1, 24, 60, fft2 // 4 + 1):
            a = world.code_spectral_envelope(make(world, sp2), fs2, fft2, d, f0_lengths=lens)
            world.synchronize()
            a = to_np(a)
            want = [ref.code_spectral_envelope(sp2[u, :lens[u]], fs2, fft2, d) for u in range(2)]
            back = np.zeros((3, 9, d))
            for u in range(2):
                assert_close_signed(a[u, :lens[u]], want[u], f"CodeSpectralEnvelope fs={fs2} d={d} utt {u}")
                assert not a[u, lens[u]:].any()                # padded frames are never written
                back[u, :lens[u]] = a[u, :lens[u]]
            assert not a[2].any()
            b = world.decode_spectral_envelope(make(world, back), fs2, fft2, d, f0_lengths=lens)
            world.synchronize()
            for u in range(2):
                assert_close(to_np(b)[u, :lens[u]], ref.decode_spectral_envelope(back[u, :lens[u]], fs2, fft2, d),
                             f"DecodeSpectralEnvelope fs={fs2} d={d} utt {u}")
        if n_ap > 0:
            a = world.code_aperiodicity(make(world, ap2), fs2, fft2, f0_lengths=lens)
            world.synchronize()
            coded = np.zeros((3, 9, n_ap))
            for u in range(2):
                coded[u, :lens[u]] = ref.code_aperiodicity(ap2[u, :lens[u]], fs2, fft2)
                assert_close_signed(to_np(a)[u, :lens[u]], coded[u, :lens[u]], f"CodeAperiodicity fs={fs2} utt {u}")
        else:
            coded = np.zeros((3, 9, 1))
        b = world.decode_aperiodicity(make(world, coded), fs2, fft2, f0_lengths=lens)
        world.synchronize()
        for u in range(2):
            want_ap = ref.decode_aperiodicity(coded[u, :lens[u]], fs2, fft2)
            assert_close(to_np(b)[u, :lens[u]], want_ap, f"DecodeAperiodicity fs={fs2} utt {u}")


def check_coded_frame_kernels(world, ref, golden):
    """CheapTrick + CodeSpectralEnvelope / D4C + CodeAperiodicity fused into the frame kernels: against the golden
    coded rows, against the two-step path of the same library (full rows, then the codec kernels), and -- other
    rates, dimensions, ragged rows, unvoiced and noise frames -- against the compiled reference's two calls."""
    x, fs = wav_from_golden(golden)
    fft, dims = int(golden["fft_size"]), int(golden["coded_dims"])
    xb = make(world, x[None, :])
    t = make(world, golden["time_axis"][None, :])
    f0 = make(world, golden["f0_stonemask"][None, :])
    opt = world.cheaptrick_option(fs)
    csp = world.cheaptrick_coded(xb, fs, t, f0, dims, opt)
    cap = world.d4c_coded(xb, fs, t, f0, fft)
    two_sp = world.code_spectral_envelope(world.cheaptrick(xb, fs, t, f0, opt), fs, fft, dims)
    two_ap = world.code_aperiodicity(world.d4c(xb, fs, t, f0, fft), fs, fft)
    world.synchronize()
    assert_close_signed(csp[0], golden["coded_sp"], "fused coded spectral envelope (golden)")
    assert_close_signed(cap[0], golden["coded_ap"], "fused coded aperiodicity (golden)")
    assert_close_signed(csp[0], to_np(two_sp)[0], "fused vs two-step coded spectral envelope", tol=1e-9)
    assert_close_signed(cap[0], to_np(two_ap)[0], "fused vs two-step coded aperiodicity", tol=1e-9)
    for fs2, n2, d2, seed in [(16000, 9000, 24, 5), (48000, 20000, 60, 6), (8000, 5000, 1, 7), (44100, 15000, 513, 8),
                              (22050, 9000, 40, 9)]:
        rng = np.random.default_rng(seed)
        tt = np.arange(n2) / fs2
        sig = 0.4 * np.sin(2 * np.pi * 180.0 * tt * (1 + 0.2 * tt)) + 0.2 * np.sin(2 * np.pi * 360.0 * tt)
        sig[n2 // 2:] = 0.0
        xs = np.stack([sig + 1e-3 * rng.normal(size=n2), 0.1 * rng.normal(size=n2)])
        lens = [n2, n2 - 1234]
        opt2 = world.cheaptrick_option(fs2)
        fft2 = opt2.fft_size
        d2 = min(d2, fft2 // 4 + 1)
        frames = [int(1000.0 * l / fs2 / 5.0) + 1 for l in lens]
        L = max(frames)
        tb, fb = np.zeros((2, L)), np.zeros((2, L))
        for u in range(2):
            tb[u, :frames[u]] = np.arange(frames[u]) * 0.005
            fb[u, :frames[u]] = np.where(rng.uniform(size=frames[u]) < 0.75, rng.uniform(60, 500, size=frames[u]), 0.0)
        a = world.cheaptrick_coded(make(world, xs), fs2, make(world, tb), make(world, fb), d2, opt2, x_lengths=lens,
                                   f0_lengths=frames)
        b = world.d4c_coded(make(world, xs), fs2, make(world, tb), make(world, fb), fft2, x_lengths=lens,
                            f0_lengths=frames)
        world.synchronize()
        a, b = to_np(a), to_np(b)
        n_ap = ref.number_of_aperiodicities(fs2)
        for u in range(2):
            xu, tu, fu = xs[u, :lens[u]], tb[u, :frames[u]], fb[u, :frames[u]]
            sp = ref.cheaptrick(xu, fs2, tu, fu)
            want = ref.code_spectral_envelope(sp, fs2, fft2, d2)
            assert_close_signed(a[u, :frames[u]], want, f"fused coded sp fs={fs2} d={d2} utt {u}")
            assert not a[u, frames[u]:].any()
            if n_ap > 0:
                ap = ref.d4c(xu, fs2, tu, fu, fft2)
                assert_close_signed(b[u, :frames[u]], ref.code_aperiodicity(ap, fs2, fft2),
                                    f"fused coded ap fs={fs2} utt {u}")
                assert not b[u, frames[u]:].any()
        if n_ap == 0:
            assert not b.any()                                  # nothing is written below 12 kHz


def wav_image(pcm_bytes, fs, nbit, extra_chunk=b""):
    """RIFF/WAVE image like the reference's wavwrite (tools/audioio.cpp:121-171), optionally with
    another chunk between fmt and data (the case wavread's scan for "data" exists for)."""
    import struct
    fmt = struct.pack("<4sIHHIIHH", b"fmt ", 16, 1, 1, fs, fs * nbit // 8, nbit // 8, nbit)
    body = b"WAVE" + fmt + extra_chunk + b"data" + struct.pack("<I", len(pcm_bytes)) + pcm_bytes
    return b"RIFF" + struct.pack("<I", len(body)) + body


def check_ingest(world, golden, ref=None, tmp_path=None):
    pcm16 = np.ascontiguousarray(golden["pcm"])
    fs = int(golden["fs"])
    # WAV header walk
    for extra in (b"", b"LIST" + (10).to_bytes(4, "little") + b"INFOdummy!"):
        img = wav_image(pcm16.tobytes(), fs, 16, extra)
        got = world.wav_parse(img)
        assert got[:3] == (fs, 16, len(pcm16)) and img[got[3]:got[3] + 4] == pcm16.tobytes()[:4]
        if ref is not None and ref.has_codec and tmp_path is not None:
            p = os.path.join(str(tmp_path), "a.wav")
            open(p, "wb").write(img)
            xr, fsr, nbit = ref.wavread(p)
            assert (fsr, nbit, len(xr)) == got[:3]
    for bad in (b"RIFX" + bytes(60), wav_image(b"", fs, 16)[:30], wav_image(pcm16.tobytes(), fs, 16).replace(b"fmt ", b"fmtx")):
        try:
            world.wav_parse(bad)
            raise AssertionError("malformed WAV accepted")
        except Exception as e:
            assert "WAV" in str(e)
    # sample conversion: exact for every width, ragged rows untouched beyond their length
    rng = np.random.default_rng(5)
    for nbit in (8, 16, 24, 32):
        nb = nbit // 8
        raw = rng.integers(0, 256, size=(3, 1000 * nb), dtype=np.uint8)
        raw[0, :nb] = 0
        raw[0, nb:2 * nb] = 255                                   # -1 LSB
        raw[0, 2 * nb:3 * nb - 1] = 0; raw[0, 3 * nb - 1] = 128   # most negative
        raw[0, 3 * nb:4 * nb - 1] = 255; raw[0, 4 * nb - 1] = 127 # most positive
        lens = [1000, 999, 1]
        x = world.pcm_to_double(make(world, raw, dtype=np.uint8), nbit, x_lengths=lens)
        world.synchronize()
        vals = np.zeros((3, 1000), dtype=np.int64)
        for j in range(nb):
            vals += raw[:, j::nb].astype(np.int64) << (8 * j)
        vals = np.where(vals >= 1 << (nbit - 1), vals - (1 << nbit), vals)
        want = vals.astype(np.float64) / float(1 << (nbit - 1))
        for u in range(3):
            assert np.array_equal(to_np(x)[u, :lens[u]], want[u, :lens[u]])
            assert not to_np(x)[u, lens[u]:].any()
        assert want[0, 2] == -1.0 and want[0, 1] == -1.0 / (1 << (nbit - 1))
    x = world.pcm_to_double(make(world, pcm16[None].view(np.uint8), dtype=np.uint8), 16)
    world.synchronize()
    assert np.array_equal(to_np(x)[0], wav_from_golden(golden)[0])


def check_analyze_coded(world, golden, f0_method=0):
    """int16 in, coded rows out, through the one-call host API; against the goldens of the DIO path."""
    import numpy as np
    pcm16 = np.ascontiguousarray(golden["pcm"])
    fs, dims = int(golden["fs"]), int(golden["coded_dims"])
    n = 3
    stride = len(pcm16) + 64
    rows = np.zeros((n, stride), dtype=np.int16)
    lens = [len(pcm16), len(pcm16) - 777, len(pcm16)]
    for u in range(n):
        rows[u, :lens[u]] = pcm16[:lens[u]]
    opt = world.analysis_option(fs, f0_method)
    t, f0, csp, cap, fl = world.analyze_coded_host(rows, 16, fs, opt, dims, x_lengths=lens)
    for u in (0, 2):
        assert fl[u] == len(golden["time_axis"])
        assert np.array_equal(t[u, :fl[u]], golden["time_axis"])
        assert_close(f0[u, :fl[u]], golden["f0_stonemask"], "f0 via analyze_coded_host")
        assert_close_signed(csp[u, :fl[u]], golden["coded_sp"], "coded sp via analyze_coded_host")
        assert_close_signed(cap[u, :fl[u]], golden["coded_ap"], "coded ap via analyze_coded_host")
    assert fl[1] < fl[0] and not csp[1, fl[1]:].any()
    # and the same call on doubles (nbit 0) gives the same numbers
    xd = rows.astype(np.float64) / 32768.0
    t2, f02, csp2, cap2, _ = world.analyze_coded_host(xd, 0, fs, opt, dims, x_lengths=lens)
    assert np.array_equal(csp2, csp) and np.array_equal(cap2, cap) and np.array_equal(f02, f0)


def check_host_pipeline_chunking(world, golden, f0_method=0):
    """analyze_host / analyze_coded_host with tiny outer / sub chunks (several outer chunks, ring slots
    reused, ragged last chunks) must give exactly what one big chunk gives."""
    pcm16 = np.ascontiguousarray(golden["pcm"])
    fs, dims = int(golden["fs"]), 24
    n, keep = 7, 6000
    rows = np.zeros((n, keep), dtype=np.int16)
    lens = [keep - 311 * u for u in range(n)]
    for u in range(n):
        rows[u, :lens[u]] = pcm16[2000 + 97 * u: 2000 + 97 * u + lens[u]]
    xd = rows.astype(np.float64) / 32768.0
    opt = world.analysis_option(fs, f0_method)
    saved = {k: os.environ.get(k) for k in ("WB_HOST_SUB", "WB_HOST_CHUNK", "WB_HOST_TAPER_MIN", "WB_HOST_TAPER")}
    try:
        for k in saved:
            os.environ.pop(k, None)
        want_raw = world.analyze_host(xd, fs, opt, x_lengths=lens)
        want_cod = world.analyze_coded_host(rows, 16, fs, opt, dims, x_lengths=lens)
        # (4, 4, 1): the last outer chunk (3 utterances) runs in quarter-size sub-chunks, the first in one
        for sub, outer, taper_min in ((1, 2, 16), (2, 4, 16), (3, 3, 16), (4, 4, 1), (4, 8, 1)):
            os.environ["WB_HOST_SUB"], os.environ["WB_HOST_CHUNK"] = str(sub), str(outer)
            os.environ["WB_HOST_TAPER_MIN"] = str(taper_min)
            got_raw = world.analyze_host(xd, fs, opt, x_lengths=lens)
            got_cod = world.analyze_coded_host(rows, 16, fs, opt, dims, x_lengths=lens)
            for a, b in zip(got_raw[:4] + got_cod[:4], want_raw[:4] + want_cod[:4]):
                assert np.array_equal(a, b), (sub, outer)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    assert (want_raw[1] > 0).any() and np.isfinite(want_raw[2]).all()


def check_analyze_batch(world, golden):
    """world_b200_analyze_batch (whole chain, device arrays, utterance slices on two internal streams) must give
    exactly what the separate stage calls give, for both F0 front ends and for every slice count."""
    pcm16 = np.ascontiguousarray(golden["pcm"])
    fs = int(golden["fs"])
    n, keep = 7, 7000
    x = np.zeros((n, keep))
    lens = [keep - 403 * u for u in range(n)]
    for u in range(n):
        x[u, :lens[u]] = pcm16[1500 + 211 * u: 1500 + 211 * u + lens[u]].astype(np.float64) / 32768.0
    xd = make(world, x)
    saved = os.environ.get("WB_LANE_SLICES")
    try:
        for method in (0, 1):
            opt = world.analysis_option(fs, method)
            if method == 1:
                t, f0, fl = world.harvest(xd, fs, opt.harvest, x_lengths=lens)
            else:
                t, f0, fl = world.dio(xd, fs, opt.dio, x_lengths=lens)
                f0 = world.stonemask(xd, fs, t, f0, x_lengths=lens, f0_lengths=fl)
            sp = world.cheaptrick(xd, fs, t, f0, opt.cheaptrick, x_lengths=lens, f0_lengths=fl)
            ap = world.d4c(xd, fs, t, f0, opt.cheaptrick.fft_size, x_lengths=lens, f0_lengths=fl)
            world.synchronize()
            want = [to_np(a).copy() for a in (t, f0, sp, ap)]
            for slices in (1, 2, 5, 8):   # 8 > n: capped to n; from 6 slices on the slices taper
                os.environ["WB_LANE_SLICES"] = str(slices)
                got = world.analyze_batch(xd, fs, opt, x_lengths=lens)
                world.synchronize()
                assert got[4] == fl
                for g, w_ in zip(got[:4], want):
                    g = to_np(g)
                    for u in range(n):   # rows beyond an utterance's frames are never written by either path
                        assert np.array_equal(g[u, :fl[u]], w_[u, :fl[u]]), (method, slices, u)
            assert (want[1] > 0).any()
    finally:
        if saved is None:
            os.environ.pop("WB_LANE_SLICES", None)
        else:
            os.environ["WB_LANE_SLICES"] = saved


def check_event_dense_and_degenerate_bands(world, ref):
    """Found by tests/fuzz/fuzz_emu_parity.py: (1) a loud tone gives every Harvest band far more zero crossings than
    its centre frequency suggests -- the per-band event lists wrap (history rings) instead of overflowing;
    (2) DIO bands above the decimated Nyquist have a zero-length window in the reference and contribute no
    candidate instead of being an error."""
    fs = 22050
    n = 19000
    t = np.arange(n) / fs
    rng = np.random.default_rng(3)
    x = np.ascontiguousarray(0.3 * np.sin(2 * np.pi * 523.0 * t) + 1e-4 * rng.normal(size=n))
    o = world.harvest_option(); o.frame_period = 1.0
    ro = ref.harvest_option(); ro.frame_period = 1.0
    # WB_EDGE_CAP_MIN shrinks the rings to the 2.5 x band frequency estimate (150 entries for the 40 Hz band
    # here, against ~450 crossings of the leaking tone), so this short signal wraps them several times
    saved = os.environ.get("WB_EDGE_CAP_MIN")
    os.environ["WB_EDGE_CAP_MIN"] = "64"
    try:
        tt, f0, fl = world.harvest(make(world, x[None]), fs, o)
        world.synchronize()
    finally:
        if saved is None:
            os.environ.pop("WB_EDGE_CAP_MIN", None)
        else:
            os.environ["WB_EDGE_CAP_MIN"] = saved
    tr, fr = ref.harvest(x, fs, ro)
    assert np.array_equal(to_np(tt)[0], tr)
    assert not ((to_np(f0)[0] > 0) != (fr > 0)).any()      # (the reference calls a bare sinusoid unvoiced)
    assert_close(to_np(f0)[0], fr, "Harvest on a loud tone (event rings wrap)")
    fs = 8000
    from synth import synth_batch
    x = synth_batch([91], fs, 4000).numpy()
    o = world.dio_option(); o.speed = 12; o.f0_ceil = 1000.0
    ro = ref.dio_option(); ro.speed = 12; ro.f0_ceil = 1000.0
    tt, f0, fl = world.dio(make(world, x), fs, o)
    world.synchronize()
    tr, fr = ref.dio(x[0], fs, ro)
    assert np.array_equal(to_np(tt)[0], tr)
    assert not ((to_np(f0)[0] > 0) != (fr > 0)).any()


def check_zero_tail_f0(world, ref):
    """SURVEY 8d: utterances that end in 0.5 s of exact zeros.  The F0 estimators must call the tail unvoiced like
    the reference does (the near-Nyquist ripple of its spectral mirroring loop is all that is left there and
    gives it a zero crossing every sample or two; the library adds the same ripple, see nyquist_bins_kernel) -- no V/UV
    flip, values within the tolerance."""
    from synth import synth_batch
    for fs, n, zt, seeds in ((16000, 24000, 8000, [1, 4]), (16000, 40000, 8000, [6]), (22050, 33075, 11025, [5])):
        x = synth_batch(seeds, fs, n, zero_tail=zt).numpy()
        xb = make(world, x)
        td, fd, fl = world.dio(xb, fs)
        th, fh, _ = world.harvest(xb, fs)
        world.synchronize()
        for u in range(len(seeds)):
            for name, t, f, (tr, fr) in (("dio", td, fd, ref.dio(x[u], fs)), ("harvest", th, fh, ref.harvest(x[u], fs))):
                got = to_np(f)[u, :fl[u]]
                assert np.array_equal(to_np(t)[u, :fl[u]], tr)
                assert not ((got > 0) != (fr > 0)).any(), f"{name}: V/UV flips in the zero tail (fs {fs}, seed {seeds[u]})"
                assert_close(got, fr, f"{name} f0 with a zero tail (fs {fs}, seed {seeds[u]})")
                assert not fr[-int(0.4 * zt / fs * 200):].any()


def check_mirroring_ripple_cases(world, ref):
    """The two situations where the reference's spectral mirroring loop (dio.cpp:319-328, harvest.cpp:122-135)
    decides its output and the library has to add the same ripple: DIO decimated to <= 2 kHz (4..12-tap band
    windows), and digital silence reaching Harvest's band filters undecimated (8 kHz input)."""
    from synth import synth_batch
    for fs, n, seed, speed, ceil in ((11025, 7502, 9, 10, 800.0), (16000, 12300, 33, 10, 1000.0), (16000, 10435, 23, 12, 400.0),
                                     (8000, 4280, 35, 12, 800.0), (16000, 13859, 43, 8, 800.0)):
        x = synth_batch([seed], fs, n).numpy()
        o = world.dio_option(); o.speed = speed; o.f0_ceil = ceil
        ro = ref.dio_option(); ro.speed = speed; ro.f0_ceil = ceil
        t, f0, fl = world.dio(make(world, x), fs, o)
        world.synchronize()
        tr, fr = ref.dio(x[0], fs, ro)
        assert np.array_equal(to_np(t)[0], tr)
        assert_close(to_np(f0)[0], fr, f"DIO fs {fs} speed {speed}")
        assert (fr > 0).sum() > 20
    rng = np.random.default_rng(11)
    for case in range(4):
        fs, n = 8000, int(rng.uniform(0.5, 1.0) * 8000)
        x = synth_batch([int(rng.integers(1, 1 << 30))], fs, n).numpy()
        a, b = sorted(rng.integers(0, n, size=2))
        x[0, a:b] = 0.0
        if case % 2 == 0:
            x[0, int(0.7 * n):] = 0.0
        t, f0, fl = world.harvest(make(world, x), fs)
        world.synchronize()
        tr, fr = ref.harvest(x[0], fs)
        got = to_np(f0)[0]
        assert not ((got > 0) != (fr > 0)).any(), f"Harvest, digital silence at 8 kHz, case {case}: V/UV flips"
        assert_close(got, fr, f"Harvest, digital silence at 8 kHz, case {case}")


def check_dio_silence_onset_bound(world, ref):
    """The one deviation class the fuzz campaigns found (DESIGN.md 6): DIO on a signal that falls into embedded DIGITAL
    silence.  On the one to four frames where the band-filtered signal decays into the silence the reference's
    candidates are set by its whole-utterance FFT rounding (~1e-17 of the signal), which a tile-wise time-domain
    filter cannot reproduce; everywhere else -- silence included, thanks to the mirroring-loop ripple -- the contour
    matches to 1e-6.  This pins the class: no V/UV flip anywhere, 1e-6 outside the onset, 1e-3 on at most six frames
    around it."""
    from synth import synth_batch
    worst_in = 0.0
    for fs, seed, a, b, speed in ((48000, 77, 8533, 27619, 2), (16000, 78, 3000, 9000, 1), (44100, 79, 9000, 30000, 4)):
        n = int(0.65 * fs)
        x = synth_batch([seed], fs, n).numpy()[0]
        x[a:b] = 0.0
        x = np.ascontiguousarray(x)
        o = world.dio_option(); ro = ref.dio_option()
        for q in (o, ro):
            q.speed = speed; q.f0_floor = 40.0; q.f0_ceil = 400.0
        t, f0, fl = world.dio(make(world, x[None]), fs, o)
        world.synchronize()
        tr, fr = ref.dio(x, fs, ro)
        got = to_np(f0)[0]
        assert np.array_equal(to_np(t)[0], tr)
        assert not ((got > 0) != (fr > 0)).any(), f"V/UV flip, fs {fs}"
        e = rel_err(got, fr)
        onset = int(a / fs / 0.005)
        near = np.zeros(len(e), dtype=bool)
        near[max(0, onset - 1):onset + 5] = True
        assert e[~near].max() <= TOL, f"fs {fs}: {e[~near].max():.2e} away from the onset of the silence"
        assert e[near].max() <= 1e-3, f"fs {fs}: {e[near].max():.2e} at the onset of the silence"
        worst_in = max(worst_in, e[near].max())
    return worst_in
