"""The exact CORE-A checker (oracle.check_corea / check_corea_ranks) and the oracle's key ranks, without a GPU.

The checker holds scores to 6e-14 absolute of |ln rd - ln rk| over the exact half-integer ranks.  These tests show
that it rejects a key rank off by one half even where the old `rtol 1e-6` bar did not, that it accepts the last-bit
differences of log(), and that the oracle ranks the keys as the reference does, ref32 wrap ties included."""
import numpy as np
import pytest
from scipy.stats import rankdata

from conftest import corea_case_names, load_corea_case


def _scores(rd, rk):
    return np.abs(np.log(rd) - np.log(rk))


@pytest.mark.parametrize("r", [1e3, 1e6, 2.0 ** 31])
def test_checker_rejects_a_key_rank_off_by_half(oracle_mod, r):
    # a class of two vertices at key rank r with scores near ln 3, among a few others
    rd = np.array([3 * r, 3 * r, 1.0, 2.5, 2.5, 7.0])
    rk = np.array([r, r, 2.0, 1.0, 1.0, 4.5])
    exact = _scores(rd, rk)
    oracle_mod.check_corea_ranks(exact, rd, rk)
    off = _scores(rd, np.where(rk == r, rk + 0.5, rk))
    assert abs(off[0] - exact[0]) > 1e-10
    with pytest.raises(AssertionError, match="off by more than"):
        oracle_mod.check_corea_ranks(off, rd, rk)
    if r >= 1e6:   # the relative bar the suite used before lets this rank bug through
        np.testing.assert_allclose(off, exact, rtol=1e-6, atol=1e-12)
    else:
        with pytest.raises(AssertionError):
            np.testing.assert_allclose(off, exact, rtol=1e-6, atol=1e-12)


def test_checker_accepts_log_rounding_and_rejects_split_ties(oracle_mod):
    rng = np.random.default_rng(0)
    n = 10_000
    rd = rng.integers(2, 2 * 2 ** 32 - 1, n) / 2.0          # half-integers up to 2^32
    rk = rng.integers(2, 2 * 2 ** 32 - 1, n) / 2.0
    rd[:100], rk[:100] = rd[0], rk[0]                       # one class of a hundred vertices
    exact = _scores(rd, rk)
    # log() one ulp off in either direction for every vertex (the same for a whole rank pair)
    la = np.nextafter(np.log(rd), np.inf)
    lb = np.nextafter(np.log(rk), -np.inf)
    oracle_mod.check_corea_ranks(np.abs(la - lb), rd, rk)
    oracle_mod.check_corea_ranks(exact, rd, rk)
    split = exact.copy()
    split[57] = np.nextafter(split[57], np.inf)             # one member of the class differs in the last bit
    with pytest.raises(AssertionError, match="share the rank pair"):
        oracle_mod.check_corea_ranks(split, rd, rk)
    nan = exact.copy()
    nan[3] = np.nan
    with pytest.raises(AssertionError):
        oracle_mod.check_corea_ranks(nan, rd, rk)


@pytest.mark.parametrize("name", corea_case_names())
def test_reference_scores_meet_the_exact_bar(oracle_mod, name):
    """The reference's own scores (glibc log) and the oracle's pass the checker: 6e-14 is not tighter than log()."""
    core, deg, ref = load_corea_case(name)
    oracle_mod.check_corea(ref, core, deg, oracle_mod.KEY_REF32)
    oracle_mod.check_corea(oracle_mod.corea(core, deg, oracle_mod.KEY_REF32), core, deg, oracle_mod.KEY_REF32)


def _keys(core, deg, mode, oracle_mod):
    k = core.astype(np.int64) * core.shape[0] + deg.astype(np.int64)
    if mode == oracle_mod.KEY_REF32:
        k = (k & 0xFFFFFFFF).astype(np.uint32).view(np.int32)
    return k


def _desc_ranks(x):
    return x.shape[0] + 1 - rankdata(x, method="average")


@pytest.mark.parametrize("mode", [0, 1])
def test_oracle_ranks_are_rankdata_of_the_keys(oracle_mod, mode):
    """Oracle key ranks = descending average ranks of the int32 (ref32, wrapped) or int64 (exact64) keys; ref32 keys
    that wrap to the same int32 are ties although their (coreness, degree) differ."""
    n = 2 ** 21
    rng = np.random.default_rng(1)
    core = rng.integers(0, 10, n).astype(np.int32)
    deg = (core + rng.integers(0, 90, n)).astype(np.int32)
    core[:1000], deg[:1000] = 2049, 50          # 2049 * 2^21 + 50 wraps to 1 * 2^21 + 50
    core[1000:2000], deg[1000:2000] = 1, 50
    core[2000:2100], deg[2000:2100] = 1099, 1099  # negative ref32 keys
    rd, rk = oracle_mod.corea_ranks(core, deg, mode)
    assert np.array_equal(rd, _desc_ranks(deg))
    assert np.array_equal(rk, _desc_ranks(_keys(core, deg, mode, oracle_mod)))
    if mode == oracle_mod.KEY_REF32:
        assert rk[0] == rk[1500] and rk[2050] == n - 49.5                 # wrapped tie; the 100 lowest keys
    else:
        assert rk[0] == 500.5 and rk[2050] == 1050.5 and rk[1500] > 1100      # the highest keys


@pytest.mark.parametrize("mode", [0, 1])
def test_oracle_ranks_with_wrapping_and_large_degrees(oracle_mod, mode):
    rng = np.random.default_rng(2)
    n = 5000
    core = rng.integers(0, 2 ** 31, n).astype(np.int32)
    deg = rng.integers(0, 2 ** 31, n).astype(np.int32)
    core[:50], deg[:50] = 7, 123
    core[50:100], deg[50:100] = 7 + 2 ** 29, 123     # 2^29 * 5000 = 0 mod 2^32: the same ref32 key
    rd, rk = oracle_mod.corea_ranks(core, deg, mode)
    keys = _keys(core, deg, mode, oracle_mod)
    assert np.array_equal(rk, _desc_ranks(keys)) and np.array_equal(rd, _desc_ranks(deg))
    assert (rk[0] == rk[75]) == (mode == oracle_mod.KEY_REF32)


def test_exact64_orders_by_the_key_for_degrees_at_least_n(oracle_mod):
    """exact64 ranks coreness * n + degree in int64, not the pair (coreness, degree): a degree >= n outranks a higher
    coreness."""
    core = np.array([0, 1, 0, 0], np.int32)
    deg = np.array([5, 0, 1, 2], np.int32)
    score = oracle_mod.corea(core, deg, oracle_mod.KEY_EXACT64)
    np.testing.assert_allclose(score, [0.0, np.log(2), np.log(4 / 3), np.log(3 / 2)], rtol=0, atol=1e-15)
    rd, rk = oracle_mod.corea_ranks(core, deg, oracle_mod.KEY_EXACT64)
    assert rk.tolist() == [1.0, 2.0, 4.0, 3.0] and rd.tolist() == [1.0, 4.0, 3.0, 2.0]
