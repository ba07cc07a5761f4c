"""Option tally_batches without a device: the history kernel's pid -> batch map (evaluated on the
host by the library itself) reproduces the contiguous particle ranges of decks.shard_range, and
the option's values are checked on the host."""
import numpy as np

from neutral_b200.decks import shard_range
from neutral_b200.host import NB200_BAD_OPTION


def _ranges_of(lib, n, B, pids):
    return np.array([lib.nb200_selftest_batch_of(int(p), n, B) for p in pids])


def _check_partition(lib, n, B):
    """Every batch's first and last pid, and their neighbours, land where shard_range puts
    them; n small enough is checked pid by pid."""
    if n <= 5000:
        got = _ranges_of(lib, n, B, range(n))
        want = np.concatenate([np.full(shard_range(n, b, B)[1], b) for b in range(B)])
        assert np.array_equal(got, want), (n, B)
        return
    for b in range(B):
        first, count = shard_range(n, b, B)
        assert count >= 1
        assert lib.nb200_selftest_batch_of(first, n, B) == b, (n, B, b)
        assert lib.nb200_selftest_batch_of(first + count - 1, n, B) == b, (n, B, b)
        if first > 0:
            assert lib.nb200_selftest_batch_of(first - 1, n, B) == b - 1, (n, B, b)
    assert shard_range(n, B - 1, B)[0] + shard_range(n, B - 1, B)[1] == n


def test_batch_of_partitions_like_shard_range(lib):
    rng = np.random.default_rng(20261020)
    cases = [(int(rng.integers(2, 5000)), int(rng.integers(2, 65))) for _ in range(40)]
    cases += [(1000, 7), (1001, 16), (1015, 64), (64, 64), (7, 7), (2, 2), (65, 64)]  # N % B != 0, B == N
    cases += [(int(rng.integers(10**5, 2**31 - 1)), int(rng.integers(2, 65))) for _ in range(10)]
    cases += [(10**8, B) for B in (2, 7, 16, 63, 64)]
    for n, B in cases:
        B = min(B, n)
        _check_partition(lib, n, B)


def test_batch_of_rejects_what_the_kernel_never_sees(lib):
    bad = 0xFFFFFFFF
    assert lib.nb200_selftest_batch_of(10, 10, 2) == bad   # pid outside [0, n)
    assert lib.nb200_selftest_batch_of(0, 4, 5) == bad     # B > n
    assert lib.nb200_selftest_batch_of(0, 2**31, 2) == bad  # beyond the 32-bit bank
    assert lib.nb200_selftest_batch_of(0, 10, 0) == bad


def test_tally_batches_option_values(lib):
    """0 and 2..64 are accepted, 1, 65 and -1 refused, all without a device."""
    prev = lib.nb200_get_option(b"tally_batches")
    assert prev == 0
    try:
        for v in [0] + list(range(2, 65)):
            assert lib.nb200_set_option(b"tally_batches", v) != NB200_BAD_OPTION, v
            assert lib.nb200_get_option(b"tally_batches") == v
        for v in (1, 65, -1):
            assert lib.nb200_set_option(b"tally_batches", v) == NB200_BAD_OPTION, v
            assert b"tally_batches" in lib.nb200_last_error()
            assert lib.nb200_get_option(b"tally_batches") == 64
    finally:
        lib.nb200_set_option(b"tally_batches", prev)
