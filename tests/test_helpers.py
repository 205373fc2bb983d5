"""The public MATLAB-style helpers of world/matlabfunctions.h (host only) against the reference's own: bit-identical
on random inputs, including the corner cases of histc (edges below the first node, on nodes, beyond the last)."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    from world_b200 import api
    return api.load_library()


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def bind(L):
    P = C.c_void_p
    L.fftshift.argtypes = [P, C.c_int, P]
    L.histc.argtypes = [P, C.c_int, P, C.c_int, P]
    L.interp1.argtypes = [P, P, C.c_int, P, C.c_int, P]
    L.decimate.argtypes = [P, C.c_int, C.c_int, P]
    L.matlab_round.argtypes = [C.c_double]; L.matlab_round.restype = C.c_int
    L.diff.argtypes = [P, C.c_int, P]
    L.interp1Q.argtypes = [C.c_double, C.c_double, P, C.c_int, P, C.c_int, P]
    L.randn.argtypes = [P]; L.randn.restype = C.c_double
    L.randn_reseed.argtypes = [P]
    L.matlab_std.argtypes = [P, C.c_int]; L.matlab_std.restype = C.c_double
    for f in (L.fftshift, L.histc, L.interp1, L.decimate, L.diff, L.interp1Q, L.randn_reseed):
        f.restype = None
    return L


def out(fn, n, dtype=np.float64, init=0.0):
    """a fresh output buffer, filled by fn"""
    o = np.full(n, init, dtype=dtype)
    fn(o)
    return o


def test_helpers_are_bit_identical_to_the_reference(lib, ref_digests):
    """Every result is compared with the reference's own for the same input, through the SHA-256 of its bytes
    (tests/refreplay.py Digests)."""
    A = bind(lib)
    B = bind(ref_digests.live.lib) if ref_digests.live is not None else None
    chk = ref_digests.check
    rng = np.random.default_rng(7)
    for trial in range(200):
        nx = int(rng.integers(2, 40))
        x = np.sort(rng.normal(size=nx)).copy()
        if trial % 5 == 0:
            x = np.arange(nx, dtype=np.float64)                      # edges can fall exactly on nodes
        y = rng.normal(size=nx)
        ne = int(rng.integers(1, 60))
        lo, hi = (x[0] - 1, x[-1] + 1) if trial % 3 else (x[0], x[-1])
        xi = np.sort(rng.uniform(lo, hi, size=ne)).copy()
        if trial % 5 == 0:
            xi = np.sort(np.round(xi * 2) / 2).copy()
        ia = out(lambda o: A.histc(ptr(x), nx, ptr(xi), ne, ptr(o)), ne, np.int32)
        chk(f"histc {trial}", ia, lambda: out(lambda o: B.histc(ptr(x), nx, ptr(xi), ne, ptr(o)), ne, np.int32))
        ya = out(lambda o: A.interp1(ptr(x), ptr(y), nx, ptr(xi), ne, ptr(o)), ne)
        chk(f"interp1 {trial}", ya, lambda: out(lambda o: B.interp1(ptr(x), ptr(y), nx, ptr(xi), ne, ptr(o)), ne))
        # interp1Q inside the grid
        x0, dx = float(rng.normal()), float(rng.uniform(0.1, 2.0))
        q = np.sort(rng.uniform(x0, x0 + dx * (nx - 1), size=ne)).copy()
        ya = out(lambda o: A.interp1Q(x0, dx, ptr(y), nx, ptr(q), ne, ptr(o)), ne)
        chk(f"interp1Q {trial}", ya, lambda: out(lambda o: B.interp1Q(x0, dx, ptr(y), nx, ptr(q), ne, ptr(o)), ne))
        da = out(lambda o: A.diff(ptr(y), nx, ptr(o)), nx)
        chk(f"diff {trial}", da, lambda: out(lambda o: B.diff(ptr(y), nx, ptr(o)), nx))
        chk(f"matlab_std {trial}", np.float64(A.matlab_std(ptr(y), nx)), lambda: np.float64(B.matlab_std(ptr(y), nx)))
        v = float(rng.normal() * 100)
        chk(f"matlab_round {trial}", np.int64(A.matlab_round(v)), lambda: np.int64(B.matlab_round(v)))
        assert A.matlab_round(0.5) == 1 and A.matlab_round(-0.5) == -1
        n2 = 2 * int(rng.integers(1, 30))
        z = rng.normal(size=n2)
        za = out(lambda o: A.fftshift(ptr(z), n2, ptr(o)), n2)
        chk(f"fftshift {trial}", za, lambda: out(lambda o: B.fftshift(ptr(z), n2, ptr(o)), n2))
    for r in range(1, 14):                                            # 1 and 13: the all-zero default branch
        n = int(rng.integers(40, 3000))
        x = rng.normal(size=n)
        # NaN-initialised: which samples are written is part of the result (NaN bytes compare like any others)
        ya = np.full(n + 16, np.nan); A.decimate(ptr(x), n, r, ptr(ya))
        chk(f"decimate {r}", ya, lambda: out(lambda o: B.decimate(ptr(x), n, r, ptr(o)), n + 16, init=np.nan))
    sa = (C.c_uint32 * 4)()
    A.randn_reseed(sa)
    ra = np.array([A.randn(sa) for _ in range(1000)] + list(sa), dtype=np.float64)

    def theirs():
        sb = (C.c_uint32 * 4)()
        B.randn_reseed(sb)
        return np.array([B.randn(sb) for _ in range(1000)] + list(sb), dtype=np.float64)
    chk("randn 1000 draws and state", ra, theirs)
