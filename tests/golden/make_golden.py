"""Generates tests/golden/vaiueo2d{,_sp,_ap}.npz from the UNMODIFIED reference (oracle/_ref, built from
/root/reference with the reference's own flags) on the reference's only fixture,
test/vaiueo2d.wav.  Run in the build container:  python tests/golden/make_golden.py
The reference ships no expected outputs (SURVEY.md 4), so these vectors are what pins parity."""
import os
import sys
import ctypes as C

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from refworld import RefWorld, read_wav  # noqa: E402

WAV = "/root/reference/test/vaiueo2d.wav"


def main():
    ref = RefWorld()
    x, fs = read_wav(WAV)
    pcm = np.round(x * 32768.0).astype(np.int16)
    out = {"pcm": pcm, "fs": np.int32(fs)}
    # DIO + StoneMask path, default options
    t, f0_dio = ref.dio(x, fs)
    f0 = ref.stonemask(x, fs, t, f0_dio)
    ct = ref.cheaptrick_option(fs)
    sp = ref.cheaptrick(x, fs, t, f0, ct)
    ap = ref.d4c(x, fs, t, f0, ct.fft_size)
    out.update(time_axis=t, f0_dio=f0_dio, f0_stonemask=f0, sp=sp, ap=ap, fft_size=np.int32(ct.fft_size))
    # Harvest path, default options (every 4th row of sp/ap keeps the fixture small)
    th, f0_h = ref.harvest(x, fs)
    assert np.array_equal(th, t)
    sp_h = ref.cheaptrick(x, fs, th, f0_h, ct)
    ap_h = ref.d4c(x, fs, th, f0_h, ct.fft_size)
    out.update(f0_harvest=f0_h, sp_harvest_rows=sp_h[::4], ap_harvest_rows=ap_h[::4])
    # the reference demo's options (test/test.cpp:103,145): f0_floor = 40 for both estimators
    od = ref.dio_option(); od.f0_floor = 40.0
    _, f0_dio40 = ref.dio(x, fs, od)
    oh = ref.harvest_option(); oh.f0_floor = 40.0
    _, f0_h40 = ref.harvest(x, fs, oh)
    out.update(f0_dio_floor40=f0_dio40, f0_stonemask_floor40=ref.stonemask(x, fs, t, f0_dio40), f0_harvest_floor40=f0_h40)
    # randn known answers: first 32 draws after randn_reseed (matlabfunctions.cpp:237-264)
    st = (C.c_uint32 * 4)()
    ref.lib.randn_reseed(st)
    ref.lib.randn.restype = C.c_double
    out["randn_first32"] = np.array([ref.lib.randn(st) for _ in range(32)])
    # ... and draws 1_000_000 .. 1_000_007 (exercises the jump-ahead)
    st = (C.c_uint32 * 4)()
    ref.lib.randn_reseed(st)
    for _ in range(1000000):
        ref.lib.randn(st)
    out["randn_at_1e6"] = np.array([ref.lib.randn(st) for _ in range(8)])
    # codec (codec.cpp:221-324) on the DIO-path envelope / aperiodicity, 40 mel-cepstral dimensions
    dims = 40
    csp = ref.code_spectral_envelope(sp, fs, ct.fft_size, dims)
    cap = ref.code_aperiodicity(ap, fs, ct.fft_size)
    out.update(coded_dims=np.int32(dims), coded_sp=csp, coded_ap=cap,
               decoded_sp_rows=ref.decode_spectral_envelope(csp, fs, ct.fft_size, dims)[::4],
               decoded_ap_rows=ref.decode_aperiodicity(cap, fs, ct.fft_size)[::4])
    # the fixture through the reference's own wavread must be what read_wav() gives
    xr, fsr, nbit = ref.wavread(WAV)
    assert fsr == fs and nbit == 16 and np.array_equal(xr, x)
    # the full-size envelope and aperiodicity go to files of their own: every file stays below 1 MB
    for part, keys in (("_sp", ["sp"]), ("_ap", ["ap"]), ("", [k for k in out if k not in ("sp", "ap")])):
        path = os.path.join(ROOT, "tests", "golden", f"vaiueo2d{part}.npz")
        np.savez_compressed(path, **{k: out[k] for k in keys})
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
