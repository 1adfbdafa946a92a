"""TEST INFRASTRUCTURE: the arguments the exp / pow replicas (maaco_path_planing_b200/csrc/mpp_libm.cuh) are checked on,
and a ctypes front-end to libm_harness.cu, which evaluates the replica and the host's libm on the host.  The harness is
compiled with nvcc on first use into a temporary directory keyed by the sources' contents."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "libm_harness.cu")
_HDR = os.path.join(os.path.dirname(_HERE), "maaco_path_planing_b200", "csrc", "mpp_libm.cuh")
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1()
        for f in (_SRC, _HDR):
            h.update(open(f, "rb").read())
        so = os.path.join(tempfile.gettempdir(), f"libmpp_libm_harness_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                                   "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        for f in (L.replica_exp_pow, L.libm_exp_pow):
            f.restype = None
            f.argtypes = [C.c_long] + [C.c_void_p] * 4
        _lib = L
    return _lib


def _run(fn, e, x, y):
    e, x, y = (np.ascontiguousarray(a, np.float64) for a in (e, x, y))
    assert e.shape == x.shape == y.shape
    out = np.empty(2 * e.size, np.float64)
    fn(e.size, e.ctypes.data, x.ctypes.data, y.ctypes.data, out.ctypes.data)
    return out


def replica(e, x, y):
    """[exp(e0), pow(x0, y0), exp(e1), ...] from mpp_exp / mpp_pow compiled for the host."""
    return _run(lib().replica_exp_pow, e, x, y)


def host_libm(e, x, y):
    """The same from the host's libm exp / pow."""
    return _run(lib().libm_exp_pow, e, x, y)


def _ulps(v, k):
    """v and its k nearest doubles on each side, for every v."""
    v = np.asarray(v, np.float64).ravel()
    out = [v]
    lo, hi = v.copy(), v.copy()
    for _ in range(k):
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
        out += [lo, hi]
    return np.concatenate(out)


def _bits(u):
    return np.array(u, np.uint64).view(np.float64)


def random_args(n, seed):
    """n seeded arguments over the domain MAACO's tables use: exp on [-800, 0]; pow with x log-uniform on [1e-7, 1e9]
    and y uniform on [0, 64], a quarter of the y whole numbers."""
    rng = np.random.default_rng(seed)
    e = rng.uniform(-800.0, 0.0, n)
    x = np.exp(rng.uniform(np.log(1e-7), np.log(1e9), n))
    y = rng.uniform(0.0, 64.0, n)
    whole = rng.random(n) < 0.25
    y[whole] = np.floor(y[whole])
    return e, x, y


def directed_args():
    """(e, x, y) for the edges of both functions, each array of the same length (the shorter sets are repeated)."""
    rng = np.random.default_rng(1975)
    ln2 = np.log(2.0)
    # exp: multiples of ln2/128 over [-800, 0] and a few ulp around them; the overflow (ln DBL_MAX), normal-underflow
    # (ln DBL_MIN), subnormal-underflow (ln 2^-1075) thresholds and the |x| = 2^-54, 512, 1024 branch points; dense
    # subnormal results; the special values
    m = np.arange(int(-800 * 128 / ln2) - 1, 1)
    e_sets = [_ulps(m * (ln2 / 128), 2),
              _ulps([709.782712893384, -708.3964185322641, -744.4400719213812, -745.1332191019411, -745.1332191019412,
                     2.0 ** -54, -2.0 ** -54, 512.0, -512.0, 1024.0, -1024.0, 709.0, -709.0, 745.0, -746.0], 64),
              rng.uniform(-745.2, -708.3, 400_000),
              rng.uniform(-1100.0, 1100.0, 100_000),
              np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 1e300, -1e300, np.finfo(np.float64).max,
                        -np.finfo(np.float64).max, 5e-324, -5e-324, 2.2250738585072014e-308, 1e-20, -1e-20]),
              _bits([0x7ff0000000000001, 0xfff0000000000123, 0x7ff8000000000456, 0x7ff4000000000000])]
    # pow: x within 64 ulp of 1 (and exact 1), exact powers of two (subnormal ones too), x near 1e-9 .. 1e9 decades;
    # y whole numbers, halves, tiny, huge and special; results near the overflow / underflow / subnormal limits
    xs_near1 = _ulps([1.0], 64)
    pow2 = 2.0 ** np.arange(-1074, 1024, dtype=np.float64)
    decades = _ulps(10.0 ** np.arange(-9, 10, dtype=np.float64), 8)
    ys = np.concatenate([np.arange(0, 65, dtype=np.float64), np.arange(0, 64, 0.5) + 0.25, [2.5, 7.0, 60.0, 1e3],
                         [-1.0, -2.5, -7.0, 1e-20, -1e-20, 2.0 ** -66, 2.0 ** -65, 2.0 ** 62, 2.0 ** 63, 2.0 ** 64,
                          -(2.0 ** 64), 1e300, -1e300, 0.0, -0.0, np.inf, -np.inf, np.nan]])
    xy = [np.meshgrid(xs_near1, ys), np.meshgrid(pow2, ys[::4]), np.meshgrid(decades, ys)]
    px = [g[0].ravel() for g in xy]
    py = [g[1].ravel() for g in xy]
    # y log2(x) near 1024 (overflow), -1022 (normal limit) and -1075 (subnormal limit) for random x
    lx = np.exp(rng.uniform(np.log(1e-7), np.log(1e9), 200_000))
    lx = lx[np.abs(np.log2(lx)) > 1e-3]
    for t in (1024.0, -1022.0, -1050.0, -1075.0):
        yy = t / np.log2(lx)
        keep = yy > 0
        px.append(lx[keep])
        py.append(_ulps(yy[keep], 0) * (1.0 + rng.uniform(-1e-12, 1e-12, keep.sum())))
    sub = 2.0 ** -1074 * np.array([1, 2, 3, 1 << 20, (1 << 52) - 1], np.float64)
    spec_x = np.concatenate([sub, [0.0, np.inf, 1.0, np.finfo(np.float64).max, 2.2250738585072014e-308]])
    sx, sy = np.meshgrid(spec_x, ys)
    px.append(sx.ravel())
    py.append(sy.ravel())
    px.append(np.full(3, 1.0))
    py.append(_bits([0x7ff4000000000000, 0x7ff8000000000001, 0xfff0000000000001]))
    e = np.concatenate(e_sets)
    x, y = np.concatenate(px), np.concatenate(py)
    n = max(e.size, x.size)
    return np.resize(e, n), np.resize(x, n), np.resize(y, n)


def mismatches(got, want):
    """Indices (into the interleaved output) where the bits differ."""
    return np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
