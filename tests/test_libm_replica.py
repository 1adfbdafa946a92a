"""mpp_exp / mpp_pow (maaco_path_planing_b200/csrc/mpp_libm.cuh), compiled for the host, return bit for bit what the
host's libm exp / pow return: on 10^7 seeded arguments over the domain MAACO's eta'^beta tables use, on directed edge
sets (x within ulps of 1, powers of two, exp arguments at multiples of ln2/128, the overflow / underflow / subnormal
thresholds, subnormal results) and on exp's special values.  CPU only.

The replica reproduces glibc 2.39's x86-64 FMA build (what a CPU with FMA and AVX2 runs); on a host whose libm is a
different build these checks fail, and so does the assumption mpp_maaco_e01_maps rests on (MAACOBatch then builds
per-map tables on the host)."""
import numpy as np
import pytest

import libm_cases as L


def _check(e, x, y):
    got, want = L.replica(e, x, y), L.host_libm(e, x, y)
    bad = L.mismatches(got, want)
    msg = [f"{'exp' if i % 2 == 0 else 'pow'}({e[i // 2]!r} | {x[i // 2]!r}, {y[i // 2]!r}): replica {got[i]!r}, "
           f"libm {want[i]!r}" for i in bad[:10]]
    assert bad.size == 0, f"{bad.size} mismatches:\n" + "\n".join(msg)


@pytest.mark.parametrize("seed", [0, 1])
def test_replica_equals_libm_on_table_domain(seed):
    _check(*L.random_args(5_000_000, seed))


def test_replica_equals_libm_on_directed_sets():
    _check(*L.directed_args())


def test_exp_special_values():
    e = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e308, -1e308, 709.8, -745.2, 5e-324, -5e-324])
    got = L.replica(e, np.ones_like(e), np.ones_like(e))[0::2]
    want = np.array([1.0, 1.0, np.inf, 0.0, np.nan, np.inf, 0.0, np.inf, 0.0, 1.0, 1.0])
    assert np.array_equal(got, want, equal_nan=True)
    _check(e, np.ones_like(e), np.ones_like(e))
