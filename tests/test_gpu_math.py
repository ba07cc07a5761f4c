"""Device builds of the bit-exact building blocks against the host: Threefry known answers,
the (0,1] mapping, the glibc-identical log on >= 1e7 inputs, cross-section brackets."""
import ctypes as C
import math

import numpy as np
import pytest

from neutral_b200.decks import cross_section_table
from test_kat import CS_INDEX_KAT, NEGLOG_KAT, THREEFRY_KAT, UNIT_KAT

pytestmark = pytest.mark.gpu

_dp = C.POINTER(C.c_double)
_u64p = C.POINTER(C.c_uint64)


def _rng_log(lib, pkey0, master_key, counter, n):
    raw = np.zeros(2 * n, dtype=np.uint64)
    unit = np.zeros(2 * n)
    neglog = np.zeros(2 * n)
    rc = lib.nb200_selftest_rng_log(pkey0, master_key, counter, n, raw.ctypes.data_as(_u64p),
                                    unit.ctypes.data_as(_dp), neglog.ctypes.data_as(_dp))
    assert rc == 0, lib.nb200_last_error()
    return raw, unit, neglog


def test_device_threefry_known_answers(gpu_lib):
    for i, ((c0, c1, k0, k1), (o0, o1)) in enumerate(THREEFRY_KAT[:6]):
        assert c1 == 0
        raw, unit, neglog = _rng_log(gpu_lib, k0, k1, c0, 1)
        assert (int(raw[0]), int(raw[1])) == (o0, o1)
        assert unit[0] == float.fromhex(UNIT_KAT[i][0]) and unit[1] == float.fromhex(UNIT_KAT[i][1])
        if i < 4:
            assert neglog[0] == float.fromhex(NEGLOG_KAT[i])


def test_device_streams_match_the_oracle(gpu_lib, port):
    raw, unit, _ = _rng_log(gpu_lib, 1000, 3, 17, 4096)
    for i in (0, 1, 77, 4095):
        assert port.threefry(17, 0, 1000 + i, 3) == (int(raw[2 * i]), int(raw[2 * i + 1]))
        assert port.random_pair(1000 + i, 3, 17) == (unit[2 * i], unit[2 * i + 1])


def test_device_log_is_glibc_log_bitwise(gpu_lib):
    rng = np.random.default_rng(7)
    n = 4_000_000
    xs = np.concatenate([rng.random(n), 0.93 + 0.14 * rng.random(n),
                         np.exp(-45.0 * rng.random(n)),
                         np.array([1.0, 0.9375, 1.0647, 2.0 ** -65, 0.5])])
    xs = np.ascontiguousarray(xs)
    ys = np.zeros_like(xs)
    assert gpu_lib.nb200_selftest_log(xs.ctypes.data_as(_dp), ys.ctypes.data_as(_dp), len(xs)) == 0
    want = np.log(xs)   # numpy calls the same libm log for scalars; verify on a sample below
    libm = C.CDLL("libm.so.6")
    libm.log.restype = C.c_double
    libm.log.argtypes = [C.c_double]
    idx = rng.integers(0, len(xs), 20000)
    for i in idx:
        assert libm.log(float(xs[i])) == ys[i], xs[i].hex()
    # full-array comparison against the host build of the same transliteration
    host = np.array([gpu_lib.nb200_host_log(float(x)) for x in xs[::37]])
    assert np.array_equal(host.view(np.uint64), ys[::37].view(np.uint64))
    mism = np.count_nonzero(want.view(np.uint64) != ys.view(np.uint64))
    # numpy may use a SIMD log of its own; it is informative only
    print(f"device log vs numpy log: {mism} of {len(xs)} differ")


def test_device_rng_plus_log_matches_libm(gpu_lib):
    """-log(rn) for 2e6 stream values, device vs host libm (what mfp sampling consumes)."""
    libm = C.CDLL("libm.so.6")
    libm.log.restype = C.c_double
    libm.log.argtypes = [C.c_double]
    _, unit, neglog = _rng_log(gpu_lib, 0, 5, 0, 1_000_000)
    rng = np.random.default_rng(3)
    for i in rng.integers(0, len(unit), 50000):
        assert -libm.log(float(unit[i])) == neglog[i]


def test_device_cross_section_brackets(gpu_lib, port):
    keys, values = cross_section_table()
    rng = np.random.default_rng(11)
    e = np.concatenate([np.array(list(CS_INDEX_KAT.keys())),
                        10.0 ** rng.uniform(-1.99, 7.99, 20000), keys[:50], keys[-50:-1]])
    e = np.ascontiguousarray(e)
    ind = np.zeros(len(e), dtype=np.int32)
    out = np.zeros(len(e))
    rc = gpu_lib.nb200_selftest_cs(keys.ctypes.data_as(_dp), values.ctypes.data_as(_dp),
                                   len(keys), e.ctypes.data_as(_dp), len(e),
                                   ind.ctypes.data_as(C.POINTER(C.c_int)),
                                   out.ctypes.data_as(_dp))
    assert rc == 0
    for i, (en, k) in enumerate(CS_INDEX_KAT.items()):
        assert ind[i] == k
    for i in range(len(e)):
        assert ind[i] == port.cs_index(keys, float(e[i]))
        assert out[i] == port.cs_lookup(keys, values, float(e[i]))


def _adversarial_tables():
    """Tables at the edges of the staged lookup's bucket index (8192 buckets over the leading
    bits of the key range; stage.cu, cs_params_from_ends)."""
    rng = np.random.default_rng(23)
    crowd = np.unique(np.concatenate([
        1.0e3 * (1.0 + np.arange(10_000) * 1.0e-13),           # within 1e-9 of one value
        [1.0e-3, 0.5, 7.0e2, 2.0e3, 1.0e6, 1.0e8]]))            # ... and a few far keys
    one = np.float64(1.0).view(np.uint64)
    return {
        "2": np.array([0.5, 3.0]),
        "3": np.array([1.0e-2, 1.0, 1.0e8]),
        "8193": np.cumsum(rng.uniform(0.5, 1.5, 8193)),
        "50000": np.geomspace(1.0e-3, 1.0e8, 50_000),
        "crowded": crowd,
        "consecutive": (one + np.arange(3000, dtype=np.uint64)).view(np.float64),  # shift 0
        "1e-300..1e300": np.geomspace(1.0e-300, 1.0e300, 6000),
    }


@pytest.mark.parametrize("name", list(_adversarial_tables()))
def test_device_cross_section_brackets_on_adversarial_tables(gpu_lib, port, name):
    """The staged lookup (bucket index + bisection) against the plain bisection on the device
    (k_selftest_cs reports -1 where they differ) and the oracle port, bit for bit: at every key,
    one ulp either side of it, the midpoints, the ends, and outside the table (clamped)."""
    keys = np.ascontiguousarray(_adversarial_tables()[name])
    assert np.all(np.diff(keys) > 0.0)
    values = np.ascontiguousarray(np.random.default_rng(len(keys)).uniform(0.5, 2.0, len(keys)))
    e = np.concatenate([keys, np.nextafter(keys, 0.0), np.nextafter(keys, np.inf),
                        0.5 * (keys[:-1] + keys[1:]),
                        [0.0, 5e-324, 0.5 * keys[0], keys[-1] * 2.0, 1.0e308]])
    e = np.ascontiguousarray(e)
    ind = np.zeros(len(e), dtype=np.int32)
    out = np.zeros(len(e))
    rc = gpu_lib.nb200_selftest_cs(keys.ctypes.data_as(_dp), values.ctypes.data_as(_dp),
                                   len(keys), e.ctypes.data_as(_dp), len(e),
                                   ind.ctypes.data_as(C.POINTER(C.c_int)),
                                   out.ctypes.data_as(_dp))
    assert rc == 0
    assert np.count_nonzero(ind == -1) == 0, "staged and plain lookups differ"
    want_i = np.array([port.cs_index(keys, float(x)) for x in e])
    want_v = np.array([port.cs_lookup(keys, values, float(x)) for x in e])
    bad = np.flatnonzero(ind != want_i)
    assert len(bad) == 0, [(e[i].hex(), ind[i], want_i[i]) for i in bad[:5]]
    bad = np.flatnonzero(out.view(np.uint64) != want_v.view(np.uint64))
    assert len(bad) == 0, [(e[i].hex(), out[i], want_v[i]) for i in bad[:5]]


def test_reciprocal_division_is_ieee_division(gpu_lib):
    """The event loop divides by loop-invariant divisors (speed, cell mean free path) through
    their correctly rounded reciprocals with a Markstein correction step; the quotient must
    be the IEEE quotient bit for bit, over the operand ranges the decks produce and beyond."""
    rng = np.random.default_rng(99)
    n = 8_000_000
    a = np.concatenate([
        10.0 ** rng.uniform(-16, 1, n // 2) * rng.choice([-1.0, 1.0], n // 2),
        rng.random(n // 4), 10.0 ** rng.uniform(-300, 300, n // 8),
        (1.0 + rng.integers(0, 2 ** 20, n // 8) * 2.0 ** -52)])          # mantissas near 1
    b = np.concatenate([
        10.0 ** rng.uniform(-6, 31, n // 2),                              # 1/Sigma_t and speeds
        10.0 ** rng.uniform(3, 8, n // 4), 10.0 ** rng.uniform(-300, 300, n // 8),
        (2.0 - rng.integers(1, 2 ** 20, n // 8) * 2.0 ** -52)])          # mantissas near 2
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    fast, ieee = np.zeros_like(a), np.zeros_like(a)
    assert gpu_lib.nb200_selftest_div(a.ctypes.data_as(_dp), b.ctypes.data_as(_dp), len(a),
                                      fast.ctypes.data_as(_dp), ieee.ctypes.data_as(_dp)) == 0
    assert np.array_equal(ieee.view(np.uint64), (a / b).view(np.uint64))  # device == host IEEE
    assert np.array_equal(fast.view(np.uint64), ieee.view(np.uint64))


def test_straight_line_cores_are_the_ieee_operators(gpu_lib):
    """div_core / rcp_core / sqrt_core (nb_fastmath.cuh: the compiler's own fast-path sequences
    without its range branch) against `/`, `1.0/` and sqrt() on the device and against numpy on
    the host, bit for bit, over the operand range the kernels admit them for
    (2^-255 <= |v| < 2^257) - mid-range magnitudes, the scatter kinematics' ratios near 1,
    mantissas at both ends of a binade, and the extremes of the admitted range."""
    rng = np.random.default_rng(2024)
    n = 6_000_000
    def operands(seed_shift):
        r = np.random.default_rng(2024 + seed_shift)
        return np.ascontiguousarray(np.concatenate([
            10.0 ** r.uniform(-30, 30, n // 3) * r.choice([-1.0, 1.0], n // 3),
            1.0 + (r.random(n // 6) - 0.5) * 0.08,                     # e'/e of a scatter
            2.0 ** r.uniform(-254.9, 256.9, n // 6),                   # the whole admitted range
            (1.0 + r.integers(0, 2 ** 22, n // 6) * 2.0 ** -52) * 2.0 ** r.integers(-40, 40, n // 6),
            (2.0 - r.integers(1, 2 ** 22, n // 6) * 2.0 ** -52) * 2.0 ** r.integers(-40, 40, n // 6),
        ]))
    a, b = operands(0), operands(1)
    out = np.zeros(6 * len(a))
    assert gpu_lib.nb200_selftest_fastmath(a.ctypes.data_as(_dp), b.ctypes.data_as(_dp), len(a),
                                           out.ctypes.data_as(_dp)) == 0
    core_div, div, core_rcp, rcp, core_sqrt, sqrt_ = out.reshape(6, -1).view(np.uint64)
    assert np.array_equal(div, (a / b).view(np.uint64))
    assert np.array_equal(rcp, (1.0 / b).view(np.uint64))
    assert np.array_equal(sqrt_, np.sqrt(np.abs(a)).view(np.uint64))
    # quotients of admitted operands can leave the normal range only beyond 2^+-512: all finite
    assert np.array_equal(core_div, div)
    assert np.array_equal(core_rcp, rcp)
    assert np.array_equal(core_sqrt, sqrt_)
    # a numerator of exactly +0 (an energy on a grid point of the cross-section table)
    z = np.zeros(1024)
    bz = np.ascontiguousarray(10.0 ** rng.uniform(-20, 20, 1024))
    outz = np.zeros(6 * 1024)
    assert gpu_lib.nb200_selftest_fastmath(z.ctypes.data_as(_dp), bz.ctypes.data_as(_dp), 1024,
                                           outz.ctypes.data_as(_dp)) == 0
    assert not outz[:1024].view(np.uint64).any()


def test_device_sincos_is_libm_sincos(gpu_lib):
    """Device sin/cos (nb_sincos.cuh) vs the host build of the same source - itself pinned to
    libm bit for bit on the same arguments - on the inject domain and across every branch."""
    rng = np.random.default_rng(11)
    r = (rng.integers(0, 2 ** 64, size=6_000_000, dtype=np.uint64).astype(np.float64)
         * 2.0 ** -64 + 2.0 ** -65)
    xs = np.concatenate([
        2.0 * math.pi * r,                                  # theta of omp3/neutral.c:612
        (rng.random(1_000_000) - 0.5) * 20.0,
        np.ldexp(rng.random(1_000_000), -rng.integers(0, 40, 1_000_000)),
        (rng.random(1_000_000) - 0.5) * 2.0e8,
        np.array([0.126, 0.855469, 2.426265, math.pi / 2, math.pi, 2.0 * math.pi, 1e-9, 0.0]),
    ])
    hi = (xs.view(np.uint64) >> np.uint64(32)) & np.uint64(0x7FFFFFFF)
    xs = np.ascontiguousarray(xs[hi < 0x419921FB])
    bad_x = C.c_double(0.0)
    assert gpu_lib.nb200_selftest_host_sincos(xs.ctypes.data_as(_dp), len(xs),
                                              C.byref(bad_x)) == 0, bad_x.value
    hs, hc = np.zeros_like(xs), np.zeros_like(xs)
    gpu_lib.nb200_host_sincos(xs.ctypes.data_as(_dp), len(xs), hs.ctypes.data_as(_dp),
                              hc.ctypes.data_as(_dp))
    ds, dc = np.zeros_like(xs), np.zeros_like(xs)
    rc = gpu_lib.nb200_selftest_sincos(xs.ctypes.data_as(_dp), ds.ctypes.data_as(_dp),
                                       dc.ctypes.data_as(_dp), len(xs))
    assert rc == 0, gpu_lib.nb200_last_error()
    assert np.array_equal(ds.view(np.uint64), hs.view(np.uint64))
    assert np.array_equal(dc.view(np.uint64), hc.view(np.uint64))
