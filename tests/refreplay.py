"""The reference's outputs as stored vectors, so that every comparison with the unmodified reference runs without it.

A test asks the `ref` fixture for reference results exactly as it would ask the compiled reference (RefWorld).
Normally each call is answered from tests/golden/reference/<test module>/<test>.npz (plus <test>.1.npz, ... where one
file would pass 1 MB): the calls of one test are replayed in the order the test makes them.  Each replayed call must
have the arguments that were recorded -- method, scalars, options, array shapes, and, for the waveform the test itself
generates, a fingerprint of its values -- else the test fails and the vectors have to be regenerated.

    WB_REF_RECORD=1 python -m pytest tests ...   # needs oracle/_ref/libworld_ref.so (oracle/Makefile, target ref)

runs the compiled reference instead and rewrites the stored calls of every test that ran.  WB_REF_RECORD may also
name a directory to write to instead of tests/golden/reference.

What is stored: every scalar, option and one-dimensional result of up to 8192 values (f0 contours, time axes) and
every other result of up to 1024 values in full.  Of a larger two-dimensional result (frames x bins: spectrogram,
aperiodicity, coded rows) the first, middle and last frames whole and two whole bin columns (every frame of the
utterance; the columns are drawn from a seed); of a longer waveform four windows of 256 samples (start, end, two
seeded) and the 16 samples around its largest magnitude.  Such a result comes back as a numpy masked array of the
full shape in which only the stored entries are unmasked; rel_err() and the masked-array reductions compare those.

Tests that compare bytes or bits with the reference (file writers, helper functions) use Digests: the SHA-256 of
each reference result, recorded the same way, against the SHA-256 of this library's result."""
import ctypes as C
import glob
import hashlib
import json
import os
import zlib

import numpy as np

from world_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "reference")
CHUNK_VALUES = 100000          # float64 values per file: compressed, each file stays below 1 MB
_OPTIONS = {"DioOption": api.DioOption, "HarvestOption": api.HarvestOption,
            "CheapTrickOption": api.CheapTrickOption, "D4COption": api.D4COption}
# RefWorld methods whose results a test may ask for
METHODS = ("frames", "dio", "harvest", "stonemask", "cheaptrick", "d4c", "synthesis", "decimate",
           "number_of_aperiodicities", "code_aperiodicity", "decode_aperiodicity", "code_spectral_envelope",
           "decode_spectral_envelope", "wavread", "dio_option", "harvest_option", "cheaptrick_option", "d4c_option")
# methods whose first argument is the waveform, which the tests generate themselves (never a result of the library)
WAVEFORM_FIRST = ("dio", "harvest", "stonemask", "cheaptrick", "d4c", "decimate")
# functions of the reference's C API called directly (ref.lib.<name>) that take and return scalars only
LIB_SCALAR = ("GetF0FloorForCheapTrick", "GetSamplesForDIO", "GetSamplesForHarvest")


def _signature(name, args):
    """What of a call must be as recorded: scalars, option fields and array shapes (array contents other than the
    waveform may be outputs of the library under test, which are not the same bits on every run)."""
    sig = [name]
    for a in args:
        if isinstance(a, C.Structure):
            sig.append(type(a).__name__ + repr([getattr(a, f) for f, _ in a._fields_]))
        elif isinstance(a, np.ndarray):
            sig.append("array" + repr(a.shape))
        elif isinstance(a, (bytes, str)):
            sig.append("path")
        else:
            sig.append(repr(a))
    return "|".join(sig)


def _fingerprint(name, args):
    """16 evenly spaced samples and the mean magnitude of the waveform argument (None for other calls)."""
    if name not in WAVEFORM_FIRST:
        return None
    x = np.asarray(args[0], dtype=np.float64).ravel()
    return [float(v) for v in x[::max(1, x.size // 16)][:16]] + [float(np.abs(x).mean()) if x.size else 0.0]


def _same_fingerprint(a, b):
    if a is None or b is None:
        return a is b
    a, b = np.array(a), np.array(b)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= 1e-9 * max(1e-300, np.abs(b).max())))


def _test_files(node, directory):
    module = os.path.splitext(os.path.basename(str(node.fspath)))[0]
    return os.path.join(directory, module), node.name


def _kept(shape, seed):
    """The entries of a large result that are stored, as a boolean mask of its shape."""
    rng = np.random.default_rng(seed)
    if len(shape) == 1:
        n, w = shape[0], 256
        m = np.zeros(n, dtype=bool)
        for s in [0, n - w] + list(rng.integers(0, n - w, size=2)):
            m[s:s + w] = True
        return m
    rows, cols = shape[0], int(np.prod(shape[1:]))
    m = np.zeros((rows, cols), dtype=bool)
    m[[0, rows // 2, rows - 1]] = True
    m[:, rng.choice(cols, size=min(2, cols), replace=False)] = True
    return m.reshape(shape)


class _Lib:
    """ref.lib for the scalar functions of LIB_SCALAR."""

    def __init__(self, owner):
        self._owner = owner

    def __getattr__(self, name):
        if name not in LIB_SCALAR:
            raise AttributeError(f"ref.lib.{name}: only {', '.join(LIB_SCALAR)} have stored results")
        return lambda *a: self._owner._call("lib." + name, a)


class _Base:
    has_dio = has_harvest = has_f0 = has_codec = True

    def __getattr__(self, name):
        if name in METHODS:
            return lambda *args: self._call(name, args)
        raise AttributeError(name)

    @property
    def lib(self):
        return _Lib(self)


class Recorder(_Base):
    """The compiled reference; every result is kept for save()."""

    def __init__(self, real, node, directory):
        self._real = real
        self._dir, self._name = _test_files(node, directory)
        self._calls, self._vals = [], []

    def _call(self, name, args):
        res = getattr(self._real.lib, name[4:])(*args) if name.startswith("lib.") else getattr(self._real, name)(*args)
        parts = res if isinstance(res, tuple) else (res,)
        n = len(self._calls)
        self._calls.append({"sig": _signature(name, args), "fp": _fingerprint(name, args),
                            "tuple": isinstance(res, tuple),
                            "parts": [self._store(zlib.crc32(f"{self._name}/{n}/{j}".encode()), p)
                                      for j, p in enumerate(parts)]})
        return res

    def _store(self, seed, v):
        if isinstance(v, C.Structure):
            self._vals.append(np.array([getattr(v, f) for f, _ in v._fields_], dtype=np.float64))
            return {"opt": type(v).__name__}
        a = np.asarray(v)
        d = {"dtype": a.dtype.str, "shape": list(a.shape)}
        if a.ndim == 0 or a.size <= 1024 or (a.ndim == 1 and a.size <= 8192):
            self._vals.append(a.astype(np.float64).ravel())
            return d
        m = _kept(a.shape, seed)
        if a.ndim == 1:
            peak = int(np.argmax(np.abs(a)))
            d["peak"] = max(0, min(a.size - 16, peak - 8))
            m[d["peak"]:d["peak"] + 16] = True
        d["seed"] = seed
        self._vals.append(a[m].astype(np.float64))
        return d

    def save(self):
        os.makedirs(self._dir, exist_ok=True)
        for old in glob.glob(os.path.join(glob.escape(self._dir), glob.escape(self._name) + ".*npz")):
            os.remove(old)
        chunk, calls, vals, k = 0, [], [], 0
        for c in self._calls:
            for _ in c["parts"]:
                vals.append(self._vals[k])
                k += 1
            calls.append(c)
            if sum(v.size for v in vals) >= CHUNK_VALUES:
                self._write(chunk, calls, vals)
                chunk, calls, vals = chunk + 1, [], []
        if calls or chunk == 0:
            self._write(chunk, calls, vals)

    def _write(self, chunk, calls, vals):
        suffix = ".npz" if chunk == 0 else f".{chunk}.npz"
        np.savez_compressed(os.path.join(self._dir, self._name + suffix), calls=np.array(json.dumps(calls)),
                            values=np.concatenate(vals) if vals else np.zeros(0))


class Replayer(_Base):
    """The stored results of one test, in the order it asks for them."""

    def __init__(self, node, directory=GOLDEN_DIR):
        d, name = _test_files(node, directory)
        first = os.path.join(d, name + ".npz")
        if not os.path.exists(first):
            raise LookupError(f"no stored reference results for {node.nodeid} ({first}); "
                              "regenerate them with WB_REF_RECORD=1 (see tests/refreplay.py)")
        self._calls, self._n = [], 0
        chunk = 0
        while os.path.exists(os.path.join(d, name + (".npz" if chunk == 0 else f".{chunk}.npz"))):
            with np.load(os.path.join(d, name + (".npz" if chunk == 0 else f".{chunk}.npz"))) as z:
                vals, off = z["values"], 0
                for c in json.loads(str(z["calls"])):
                    c["values"] = []
                    for p in c["parts"]:
                        size = self._stored_size(p)
                        c["values"].append(vals[off:off + size])
                        off += size
                    self._calls.append(c)
            chunk += 1

    @staticmethod
    def _stored_size(p):
        if "opt" in p:
            return len(_OPTIONS[p["opt"]]._fields_)
        if "seed" not in p:
            return int(np.prod(p["shape"]))
        return int(Replayer._mask(p).sum())

    @staticmethod
    def _mask(p):
        m = _kept(tuple(p["shape"]), p["seed"])
        if "peak" in p:
            m[p["peak"]:p["peak"] + 16] = True
        return m

    def _call(self, name, args):
        n = self._n
        self._n += 1
        if n >= len(self._calls):
            raise LookupError(f"call {n} ({name}) was not made by this test when its reference results were stored")
        c, got = self._calls[n], _signature(name, args)
        if c["sig"] != got or not _same_fingerprint(_fingerprint(name, args), c["fp"]):
            raise LookupError(f"call {n}: stored reference call {c['sig']!r} (waveform {c['fp']}) but the test now "
                              f"calls {got!r} (waveform {_fingerprint(name, args)}); regenerate the stored results "
                              "(tests/refreplay.py)")
        parts = tuple(self._load(p, v) for p, v in zip(c["parts"], c["values"]))
        return parts if c["tuple"] else parts[0]

    def _load(self, p, v):
        if "opt" in p:
            o = _OPTIONS[p["opt"]]()
            for (f, ty), x in zip(o._fields_, v):
                setattr(o, f, int(x) if ty is C.c_int else float(x))
            return o
        shape, dtype = tuple(p["shape"]), np.dtype(p["dtype"])
        if "seed" not in p:
            a = v.astype(dtype).reshape(shape)
            return a.item() if a.ndim == 0 else a
        m = self._mask(p)
        data = np.full(shape, np.nan)
        data[m] = v
        return np.ma.masked_array(data.astype(dtype), mask=~m)


def _digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(a.dtype.str.encode() + repr(a.shape).encode() + a.tobytes()).hexdigest()


class Digests:
    """Bit-exact comparisons with the reference: check(what, ours, theirs) asserts that `ours` has exactly the bytes
    of the reference's result.  Recording (live reference given): `theirs()` is called and its SHA-256 stored;
    otherwise the stored SHA-256 of the same check, in the same order, is the one compared against."""

    def __init__(self, node, live=None, directory=GOLDEN_DIR):
        d, name = _test_files(node, directory)
        self._path = os.path.join(d, name + ".json")
        self.live = self._live = live
        if live is None:
            if not os.path.exists(self._path):
                raise LookupError(f"no stored reference digests for {node.nodeid} ({self._path}); "
                                  "regenerate them with WB_REF_RECORD=1 (see tests/refreplay.py)")
            with open(self._path) as f:
                self._stored = json.load(f)
        else:
            self._stored = []
        self._n = 0

    def check(self, what, ours, theirs):
        """ours: bytes or array; theirs: a function computing the reference's result (used when recording)."""
        got = hashlib.sha256(ours).hexdigest() if isinstance(ours, bytes) else _digest(ours)
        if self._live is not None:
            t = theirs()
            want = hashlib.sha256(t).hexdigest() if isinstance(t, bytes) else _digest(t)
            self._stored.append([what, want])
        else:
            assert self._n < len(self._stored), f"{what}: no stored reference digest (regenerate them)"
            assert self._stored[self._n][0] == what, f"{what}: stored digest is for {self._stored[self._n][0]}"
            want = self._stored[self._n][1]
        self._n += 1
        assert got == want, f"{what}: differs from the reference's result"

    def save(self):
        os.makedirs(os.path.dirname(self._path), exist_ok=True)
        with open(self._path, "w") as f:
            json.dump(self._stored, f, indent=0)


def load_vaiueo2d():
    """The reference's results on its fixture (tests/golden/make_golden.py), kept in three files below 1 MB each."""
    out = {}
    for part in ("", "_sp", "_ap"):
        with np.load(os.path.join(ROOT, "tests", "golden", f"vaiueo2d{part}.npz")) as z:
            out.update({k: z[k] for k in z.files})
    return out
