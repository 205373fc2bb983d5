"""ctypes access to the checkers (test infrastructure only):
  * oracle/_ref/libworld_ref.so  -- the unmodified reference compiled from /root/reference
  * oracle/libworld_oracle.so    -- our CPU restatement (oracle/world_oracle.cpp)
Both export the reference's C API, so one wrapper class serves both."""
import ctypes as C
import os
import wave

import numpy as np

from world_b200.api import DioOption, HarvestOption, CheapTrickOption, D4COption

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libworld_ref.so")
ORACLE_LIB = os.path.join(ROOT, "oracle", "libworld_oracle.so")
_P = C.c_void_p


def read_wav(path):
    """mono PCM -> float64 in [-1, 1) exactly like tools/audioio.cpp:236-249 (int / 2^(nbit-1))."""
    with wave.open(path, "rb") as w:
        assert w.getnchannels() == 1 and w.getsampwidth() == 2
        fs = w.getframerate()
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2")
    return pcm.astype(np.float64) / 32768.0, fs


class RefWorld:
    def __init__(self, path=REF_LIB):
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        # RTLD_LOCAL: these symbols have the same names as the product's legacy API
        self.lib = C.CDLL(path, mode=os.RTLD_LOCAL | os.RTLD_NOW)
        L = self.lib
        L.GetSamplesForDIO.restype = C.c_int
        L.GetSamplesForDIO.argtypes = [C.c_int, C.c_int, C.c_double]
        L.GetSamplesForHarvest.restype = C.c_int
        L.GetSamplesForHarvest.argtypes = [C.c_int, C.c_int, C.c_double]
        L.GetFFTSizeForCheapTrick.restype = C.c_int
        L.GetF0FloorForCheapTrick.restype = C.c_double
        L.GetF0FloorForCheapTrick.argtypes = [C.c_int, C.c_int]
        self.has_dio, self.has_harvest = hasattr(L, "Dio"), hasattr(L, "Harvest")  # the restatement has no Harvest
        self.has_f0 = self.has_dio and self.has_harvest
        if self.has_dio:
            L.Dio.argtypes = [_P, C.c_int, C.c_int, C.POINTER(DioOption), _P, _P]
            L.Dio.restype = None
        if self.has_harvest:
            L.Harvest.argtypes = [_P, C.c_int, C.c_int, C.POINTER(HarvestOption), _P, _P]
            L.Harvest.restype = None
        L.StoneMask.argtypes = [_P, C.c_int, C.c_int, _P, _P, C.c_int, _P]
        L.CheapTrick.argtypes = [_P, C.c_int, C.c_int, _P, _P, C.c_int, C.POINTER(CheapTrickOption), _P]
        L.D4C.argtypes = [_P, C.c_int, C.c_int, _P, _P, C.c_int, C.c_int, C.POINTER(D4COption), _P]
        for f in (L.StoneMask, L.CheapTrick, L.D4C):
            f.restype = None
        self.has_codec = hasattr(L, "CodeSpectralEnvelope")
        if self.has_codec:
            L.GetNumberOfAperiodicities.restype = C.c_int
            L.GetNumberOfAperiodicities.argtypes = [C.c_int]
            for f in (L.CodeAperiodicity, L.DecodeAperiodicity):
                f.restype = None
                f.argtypes = [_P, C.c_int, C.c_int, C.c_int, _P]
            for f in (L.CodeSpectralEnvelope, L.DecodeSpectralEnvelope):
                f.restype = None
                f.argtypes = [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P]

    # options
    def dio_option(self):
        o = DioOption(); self.lib.InitializeDioOption(C.byref(o)); return o

    def harvest_option(self):
        o = HarvestOption(); self.lib.InitializeHarvestOption(C.byref(o)); return o

    def cheaptrick_option(self, fs):
        o = CheapTrickOption(); self.lib.InitializeCheapTrickOption(C.c_int(fs), C.byref(o)); return o

    def d4c_option(self):
        o = D4COption(); self.lib.InitializeD4COption(C.byref(o)); return o

    def frames(self, fs, n, frame_period=5.0):
        return self.lib.GetSamplesForDIO(fs, n, frame_period)

    @staticmethod
    def _rows(a):
        ptrs = (C.c_void_p * a.shape[0])(*[a[i].ctypes.data for i in range(a.shape[0])])
        return ptrs

    def dio(self, x, fs, opt=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        opt = opt or self.dio_option()
        L = self.lib.GetSamplesForDIO(fs, len(x), opt.frame_period)
        t = np.zeros(L); f0 = np.zeros(L)
        self.lib.Dio(x.ctypes.data, len(x), fs, C.byref(opt), t.ctypes.data, f0.ctypes.data)
        return t, f0

    def harvest(self, x, fs, opt=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        opt = opt or self.harvest_option()
        L = self.lib.GetSamplesForHarvest(fs, len(x), opt.frame_period)
        t = np.zeros(L); f0 = np.zeros(L)
        self.lib.Harvest(x.ctypes.data, len(x), fs, C.byref(opt), t.ctypes.data, f0.ctypes.data)
        return t, f0

    def stonemask(self, x, fs, t, f0):
        x = np.ascontiguousarray(x, dtype=np.float64)
        t = np.ascontiguousarray(t); f0 = np.ascontiguousarray(f0)
        out = np.zeros_like(f0)
        self.lib.StoneMask(x.ctypes.data, len(x), fs, t.ctypes.data, f0.ctypes.data, len(f0), out.ctypes.data)
        return out

    def cheaptrick(self, x, fs, t, f0, opt=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        t = np.ascontiguousarray(t); f0 = np.ascontiguousarray(f0)
        opt = opt or self.cheaptrick_option(fs)
        sp = np.zeros((len(f0), opt.fft_size // 2 + 1))
        rows = self._rows(sp)
        self.lib.CheapTrick(x.ctypes.data, len(x), fs, t.ctypes.data, f0.ctypes.data, len(f0), C.byref(opt), rows)
        return sp

    def synthesis(self, f0, sp, ap, fft_size, frame_period, fs, y_length):
        f0 = np.ascontiguousarray(f0); sp = np.ascontiguousarray(sp); ap = np.ascontiguousarray(ap)
        y = np.zeros(y_length)
        self.lib.Synthesis.restype = None
        self.lib.Synthesis.argtypes = [_P, C.c_int, _P, _P, C.c_int, C.c_double, C.c_int, C.c_int, _P]
        self.lib.Synthesis(f0.ctypes.data, len(f0), self._rows(sp), self._rows(ap), fft_size, frame_period, fs,
                           y_length, y.ctypes.data)
        return y

    def d4c(self, x, fs, t, f0, fft_size, opt=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        t = np.ascontiguousarray(t); f0 = np.ascontiguousarray(f0)
        opt = opt or self.d4c_option()
        ap = np.zeros((len(f0), fft_size // 2 + 1))
        rows = self._rows(ap)
        self.lib.D4C(x.ctypes.data, len(x), fs, t.ctypes.data, f0.ctypes.data, len(f0), fft_size, C.byref(opt), rows)
        return ap


    # codec.h
    def number_of_aperiodicities(self, fs):
        return self.lib.GetNumberOfAperiodicities(fs)

    def _codec(self, fn, src, out_w, *args):
        src = np.ascontiguousarray(src, dtype=np.float64)
        out = np.zeros((src.shape[0], out_w))
        fn(self._rows(src), src.shape[0], *args, self._rows(out))
        return out

    def code_aperiodicity(self, ap, fs, fft_size):
        return self._codec(self.lib.CodeAperiodicity, ap, max(1, self.number_of_aperiodicities(fs)), fs, fft_size)

    def decode_aperiodicity(self, coded, fs, fft_size):
        return self._codec(self.lib.DecodeAperiodicity, coded, fft_size // 2 + 1, fs, fft_size)

    def code_spectral_envelope(self, sp, fs, fft_size, dims):
        return self._codec(self.lib.CodeSpectralEnvelope, sp, dims, fs, fft_size, dims)

    def decode_spectral_envelope(self, coded, fs, fft_size, dims):
        return self._codec(self.lib.DecodeSpectralEnvelope, coded, fft_size // 2 + 1, fs, fft_size, dims)

    def decimate(self, x, r):
        """the reference's decimate() (matlabfunctions.cpp)"""
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros(len(x))
        self.lib.decimate(x.ctypes.data_as(C.c_void_p), len(x), r, y.ctypes.data_as(C.c_void_p))
        return y

    def wavread(self, path):
        """the reference's own wavread (tools/audioio.cpp:217-252); only in oracle/_ref"""
        self.lib.GetAudioLength.restype = C.c_int
        self.lib.GetAudioLength.argtypes = [C.c_char_p]
        self.lib.wavread.restype = None
        self.lib.wavread.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), _P]
        n = self.lib.GetAudioLength(path.encode())
        x = np.zeros(max(n, 1)); fs = C.c_int(); nbit = C.c_int()
        self.lib.wavread(path.encode(), C.byref(fs), C.byref(nbit), x.ctypes.data)
        return x[:n], fs.value, nbit.value


def rel_err(got, want, floor=0.0):
    """max |got-want| / max(|want|, floor); exact zeros in `want` must be matched exactly unless floor>0.
    A masked `want` (a sampled stored result, tests/refreplay.py) is compared on its unmasked entries only."""
    known = ~np.ma.getmaskarray(want)
    got = np.asarray(got, dtype=np.float64); want = np.ma.getdata(want).astype(np.float64)
    den = np.maximum(np.abs(want), floor)
    diff = np.abs(got - want)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(den > 0, diff / den, np.where(diff == 0, 0.0, np.inf))
    return np.where(known, r, 0.0)
