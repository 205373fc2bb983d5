"""The reference's OWN example programs (examples/codec_test/*.cpp, examples/analysis_synthesis/analysis.cpp),
compiled unchanged by oracle/Makefile once against the compiled reference and once against this library's
headers and libworld_b200.so.  CPU: everything builds and links; the library-linked programs refuse to
compute without a GPU.  GPU: both chains  wav -> f0analysis (Harvest) -> spanalysis -d 40 -> apanalysis -c ->
readandsynthesis -> wav  run on the reference's fixture and the files they write are compared."""
import os
import subprocess
import wave

import numpy as np
import pytest

import test_abi
import test_parity_common as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EX = os.path.join(ROOT, "oracle", "_ref", "examples")
NAMES = ["f0analysis", "spanalysis", "apanalysis", "readandsynthesis", "analysis"]


@pytest.fixture(scope="module")
def examples():
    # the programs' sources are the reference's, so build() can only compile them where those sources are present
    if not all(os.path.exists(os.path.join(EX, f"{k}_{n}")) for k in ("ref", "b200") for n in NAMES):
        pytest.skip("oracle/_ref/examples not built (the reference's example sources were absent at build time)")
    return EX


def write_fixture_wav(golden, path):
    with wave.open(path, "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(int(golden["fs"]))
        w.writeframes(np.ascontiguousarray(golden["pcm"]).astype("<i2").tobytes())


def run_chain(ex, kind, d):
    def run(name, *args):
        r = subprocess.run([os.path.join(ex, f"{kind}_{name}"), *args], cwd=d, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        return r
    run("f0analysis", "in.wav", "-o", f"{kind}.f0")
    run("spanalysis", "in.wav", f"{kind}.f0", "-d", "40", "-o", f"{kind}.sp")
    run("apanalysis", "in.wav", f"{kind}.f0", "-c", "-o", f"{kind}.ap")
    run("readandsynthesis", f"{kind}.f0", f"{kind}.sp", f"{kind}.ap", "-o", f"{kind}.wav")
    run("analysis", "in.wav", f"{kind}_a.f0", f"{kind}_a.sp", f"{kind}_a.ap")


def read_f0_file(path):
    b = open(path, "rb").read()
    assert b[:4] == b"F0  " and b[4:8] == b"NOF " and b[12:16] == b"FP  "
    n = int.from_bytes(b[8:12], "little")
    return np.frombuffer(b[24:24 + 8 * n], dtype="<f8")


def read_rows_file(path, tag):
    b = open(path, "rb").read()
    assert b[:4] == tag
    n = int.from_bytes(b[8:12], "little"); fft = int.from_bytes(b[28:32], "little"); nod = int.from_bytes(b[36:40], "little")
    w = nod if nod else fft // 2 + 1
    return np.frombuffer(b[48:48 + 8 * n * w], dtype="<f8").reshape(n, w)


def test_reference_examples_build_unchanged_against_this_library(examples, golden, tmp_path):
    import torch
    d = str(tmp_path)
    write_fixture_wav(golden, os.path.join(d, "in.wav"))
    run_chain(examples, "ref", d)                       # the reference's programs on the reference library
    assert len(read_f0_file(os.path.join(d, "ref.f0"))) == len(golden["time_axis"])
    assert read_rows_file(os.path.join(d, "ref.sp"), b"SPEC").shape == (len(golden["time_axis"]), 40)
    if not torch.cuda.is_available():
        r = subprocess.run([os.path.join(examples, "b200_f0analysis"), "in.wav", "-o", "b.f0"], cwd=d,
                           capture_output=True, text=True, timeout=120)
        assert "no CPU path" in r.stderr                # linked against this library: no GPU, no result


@pytest.mark.gpu
def test_gpu_reference_examples_run_on_this_library(examples, golden, tmp_path):
    d = str(tmp_path)
    write_fixture_wav(golden, os.path.join(d, "in.wav"))
    run_chain(examples, "ref", d)
    run_chain(examples, "b200", d)
    p = lambda n: os.path.join(d, n)
    f_ref, f_b = read_f0_file(p("ref.f0")), read_f0_file(p("b200.f0"))
    assert not ((f_ref > 0) != (f_b > 0)).any()
    pc.assert_close(f_b, f_ref, "f0analysis (Harvest) through the reference's program")
    pc.assert_close_signed(read_rows_file(p("b200.sp"), b"SPEC"), read_rows_file(p("ref.sp"), b"SPEC"), "spanalysis -d 40")
    pc.assert_close_signed(read_rows_file(p("b200.ap"), b"AP  "), read_rows_file(p("ref.ap"), b"AP  "), "apanalysis -c")
    with wave.open(p("ref.wav")) as a, wave.open(p("b200.wav")) as b:
        ya = np.frombuffer(a.readframes(a.getnframes()), dtype="<i2").astype(np.int32)
        yb = np.frombuffer(b.readframes(b.getnframes()), dtype="<i2").astype(np.int32)
    assert len(ya) == len(yb) and np.abs(ya).max() > 1000
    assert np.abs(ya - yb).max() <= 1                   # int16 quantisation of waveforms that differ by ~1e-12
    # examples/analysis_synthesis/analysis writes raw float64 streams (DIO + StoneMask, CheapTrick, D4C)
    # (the envelope stream starts with the sampling rate as int32 and the frame period as float64)
    for ext, width, skip in (("f0", 1, 0), ("sp", int(golden["fft_size"]) // 2 + 1, 12), ("ap", int(golden["fft_size"]) // 2 + 1, 0)):
        ba, bb = open(p(f"ref_a.{ext}"), "rb").read(), open(p(f"b200_a.{ext}"), "rb").read()
        assert len(ba) == len(bb) and ba[:skip] == bb[:skip]
        ra, rb = np.frombuffer(ba[skip:], dtype="<f8"), np.frombuffer(bb[skip:], dtype="<f8")
        assert ra.size % width == 0 and ra.size > 0
        pc.assert_close(rb, ra, f"analysis example, .{ext} stream")


@pytest.mark.gpu
def test_gpu_cpp_batched_overloads_equal_single_utterance_api(tmp_path):
    exe = test_abi.build_cpp_overload_program(tmp_path / "batch_overloads")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.startswith("OK")
