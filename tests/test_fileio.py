"""File glue (SURVEY.md 8 rows f3 / f4): WAV and parameter files written by this library are byte-identical to
what the reference's tools write, and each side reads the other's files.  Host-only code: no GPU needed (the
library loads without one)."""
import ctypes as C
import os

import numpy as np
import pytest

import test_parity_common as pc


@pytest.fixture(scope="module")
def lib():
    from world_b200 import api
    return api.load_library()


def rows_of(a):
    return (C.c_void_p * a.shape[0])(*[a[i].ctypes.data for i in range(a.shape[0])])


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _bytes(path):
    with open(path, "rb") as f:
        return f.read()


def test_wav_files_match_the_reference(lib, ref_digests, golden, tmp_path):
    """The reference's files and readings are compared through their SHA-256 (tests/refreplay.py Digests).  Once a
    file of ours is checked to be byte-identical to the reference's, it stands in for the reference's file."""
    R = ref_digests.live
    x, fs = pc.wav_from_golden(golden)
    x = np.ascontiguousarray(np.concatenate([x, [1.5, -1.5, 0.99999, -1.0]]))   # clamping cases
    ours, theirs = str(tmp_path / "ours.wav").encode(), str(tmp_path / "ref.wav").encode()
    lib.wavwrite(ptr(x), len(x), fs, 16, ours)

    def ref_wav():
        R.lib.wavwrite.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p]
        R.lib.wavwrite.restype = None
        R.lib.wavwrite(ptr(x), len(x), fs, 16, theirs)
        return _bytes(theirs)
    ref_digests.check("wavwrite bytes", _bytes(ours), ref_wav)
    if R is None:
        theirs = ours
    # each reader on the other's file
    assert lib.GetAudioLength(theirs) == len(x)
    y = np.zeros(len(x)); f = C.c_int(); nb = C.c_int()
    lib.wavread(theirs, C.byref(f), C.byref(nb), ptr(y))
    assert (f.value, nb.value) == (fs, 16)

    def ref_read():
        yr, fsr, nbr = R.wavread(ours.decode())
        return np.concatenate([[fsr, nbr], yr])
    ref_digests.check("reference wavread of ours", np.concatenate([[fs, 16], y]), ref_read)
    assert lib.GetAudioLength(str(tmp_path / "missing.wav").encode()) == 0
    open(tmp_path / "bad.wav", "wb").write(b"RIFX" + bytes(60))
    assert lib.GetAudioLength(str(tmp_path / "bad.wav").encode()) == -1


def _bind_files(L_):
    L_.WriteF0.argtypes = [C.c_char_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_int]
    L_.WriteF0.restype = None
    L_.ReadF0.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p]
    L_.GetHeaderInformation.argtypes = [C.c_char_p, C.c_char_p]
    L_.GetHeaderInformation.restype = C.c_double
    for fn in (L_.WriteSpectralEnvelope, L_.WriteAperiodicity):
        fn.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p]
        fn.restype = None
    for fn in (L_.ReadSpectralEnvelope, L_.ReadAperiodicity):
        fn.argtypes = [C.c_char_p, C.c_void_p]


def test_parameter_files_match_the_reference(lib, ref_digests, golden, tmp_path):
    """As above: the reference's files and readings through their SHA-256."""
    R = ref_digests.live.lib if ref_digests.live is not None else None
    chk = ref_digests.check
    fs, fft = int(golden["fs"]), int(golden["fft_size"])
    t = np.ascontiguousarray(golden["time_axis"]); f0 = np.ascontiguousarray(golden["f0_harvest"])
    sp = np.ascontiguousarray(golden["sp"]); cap = np.ascontiguousarray(golden["coded_ap"])
    L = len(f0)
    p = lambda name: str(tmp_path / name).encode()
    _bind_files(lib)
    if R is not None:
        _bind_files(R)

    def theirs_file(write, name):
        write(p(name))
        return _bytes(p(name))
    for text in (0, 1):
        lib.WriteF0(p(f"o{text}.f0"), L, 5.0, ptr(t), ptr(f0), text)
        chk(f"WriteF0 text={text}", _bytes(p(f"o{text}.f0")),
            lambda: theirs_file(lambda q: R.WriteF0(q, L, 5.0, ptr(t), ptr(f0), text), f"r{text}.f0"))
    r0 = "r0.f0" if R is not None else "o0.f0"      # byte-identical (checked above)

    def read_f0(who, name):
        t2 = np.zeros(L); f2 = np.zeros(L)
        ok = who.ReadF0(p(name), ptr(t2), ptr(f2))
        return np.concatenate([[ok, who.GetHeaderInformation(p(name), b"NOF "), who.GetHeaderInformation(p(name), b"FP  ")],
                               t2, f2])
    want_f0 = np.concatenate([[1, L, 5.0], np.arange(L) / 1000.0 * 5.0, f0])
    assert np.array_equal(read_f0(lib, r0), want_f0)
    chk("reference ReadF0 of ours", want_f0, lambda: read_f0(R, "o0.f0"))
    # full-width envelope (NOD = 0) and coded aperiodicity (NOD = 2)
    lib.WriteSpectralEnvelope(p("o.sp"), fs, L, 5.0, fft, 0, rows_of(sp))
    lib.WriteAperiodicity(p("o.ap"), fs, L, 5.0, fft, cap.shape[1], rows_of(cap))
    chk("WriteSpectralEnvelope", _bytes(p("o.sp")),
        lambda: theirs_file(lambda q: R.WriteSpectralEnvelope(q, fs, L, 5.0, fft, 0, rows_of(sp)), "r.sp"))
    chk("WriteAperiodicity", _bytes(p("o.ap")),
        lambda: theirs_file(lambda q: R.WriteAperiodicity(q, fs, L, 5.0, fft, cap.shape[1], rows_of(cap)), "r.ap"))
    r_sp, r_ap = ("r.sp", "r.ap") if R is not None else ("o.sp", "o.ap")

    def read_rows(who, sp_file, ap_file):
        a = np.zeros_like(sp); b = np.zeros_like(cap)
        ok = [who.ReadSpectralEnvelope(p(sp_file), rows_of(a)), who.ReadAperiodicity(p(ap_file), rows_of(b))]
        heads = [who.GetHeaderInformation(p(sp_file), key) for key in (b"NOF ", b"FFT ", b"NOD ", b"FS  ")]
        return np.concatenate([ok, heads, a.ravel(), b.ravel()])
    want_rows = np.concatenate([[1, 1, L, fft, 0, fs], sp.ravel(), cap.ravel()])
    assert np.array_equal(read_rows(lib, r_sp, r_ap), want_rows)
    chk("reference ReadSpectralEnvelope / ReadAperiodicity of ours", want_rows, lambda: read_rows(R, "o.sp", "o.ap"))
    assert lib.ReadAperiodicity(p("o.sp"), rows_of(np.zeros_like(sp))) == 0          # wrong tag
    # flat-row variants used with the batched ABI's arrays
    assert lib.world_b200_write_rows(p("flat.sp"), b"SPEC", fs, L, 5.0, fft, 0, ptr(sp)) == 0
    assert _bytes(p("flat.sp")) == _bytes(p(r_sp))
    back = np.zeros_like(sp)
    assert lib.world_b200_read_rows(p(r_sp), b"SPEC", ptr(back), L) == 0 and np.array_equal(back, sp)
    assert lib.world_b200_read_rows(p(r_sp), b"SPEC", ptr(back), L - 1) != 0
    assert lib.world_b200_write_rows(p("x"), b"NOPE", fs, L, 5.0, fft, 0, ptr(sp)) != 0
