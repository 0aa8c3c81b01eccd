"""Float-descriptor extension (SURVEY 8 row a8): squared-L2 top-2 on tcgen05 vs the exact oracle.

Tolerances (north_star): indices identical except documented near-ties; distances within 1e-4 relative."""
import numpy as np
import pytest

from oracle import orc

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _check(matcher, q, t):
    bj, bd, sj, sd = matcher.knn2_l2(q, t)
    ej, ed, fj, fd = orc.l2_knn2(q, t)
    n2 = len(t)
    d = ((q[:, None, :].astype(np.float64) - t[None].astype(np.float64)) ** 2).sum(-1) if len(q) * n2 <= 4_000_000 else None
    for got_j, got_d, exp_j, exp_d in ((bj, bd, ej, ed), (sj, sd, fj, fd)):
        assert ((got_j >= 0) == (exp_j >= 0)).all()
        ok = exp_j >= 0
        np.testing.assert_allclose(got_d[ok], exp_d[ok], rtol=RTOL, atol=1e-6)       # distances: 1e-4 relative
        diff = ok & (got_j != exp_j)
        # an index may differ only at a near-tie: the chosen neighbour is as close as the oracle's within RTOL
        if diff.any():
            assert d is not None
            rows = np.nonzero(diff)[0]
            assert np.allclose(d[rows, got_j[rows]], exp_d[rows], rtol=RTOL, atol=1e-6)
            assert diff.mean() < 0.01
    return bj, bd, sj, sd


@pytest.mark.parametrize("n1,n2,dim", [(128, 128, 64), (128, 256, 128), (300, 500, 128), (1000, 777, 100),
                                        (77, 1300, 32), (5, 3, 128), (9, 1, 16), (129, 4097, 128)])
def test_l2_knn2_random(matcher, n1, n2, dim):
    rng = np.random.default_rng(n1 * 7 + n2)
    q = rng.standard_normal((n1, dim)).astype(np.float32)
    t = rng.standard_normal((n2, dim)).astype(np.float32)
    _check(matcher, q, t)
    if n1 <= 128:                                   # the single-CTA kernel ranks with the three-term bf16 split
        assert matcher.l2_last_fallback_rows() == -1


def test_l2_noisy_copies_small_distances(matcher):
    # train = query + small noise: the cancellation-prone case for ||q||^2 + ||t||^2 - 2 q.t
    rng = np.random.default_rng(5)
    q = (rng.standard_normal((2000, 128)) * 3).astype(np.float32)
    t = (q[rng.permutation(2000)] + rng.standard_normal((2000, 128)).astype(np.float32) * 0.01).astype(np.float32)
    bj, bd, _, _ = _check(matcher, q, t)
    assert bd.max() < 0.1


def test_l2_config2_shape_8k(matcher):
    rng = np.random.default_rng(11)
    q = rng.random((8192, 128), dtype=np.float32)           # SIFT-like non-negative descriptors
    t = rng.random((8192, 128), dtype=np.float32)
    _check(matcher, q, t)


def test_l2_heterogeneous_norms(matcher):
    # row norms spread over four orders of magnitude on both sides: the norms are folded into the GEMM
    # (-(|q|^2 + |t|^2)/2 rides in an extra operand chunk), so their precision must hold per pair of rows
    rng = np.random.default_rng(21)
    q = (rng.standard_normal((700, 96)) * 10.0 ** rng.uniform(-2, 2, size=(700, 1))).astype(np.float32)
    t = (rng.standard_normal((1500, 96)) * 10.0 ** rng.uniform(-2, 2, size=(1500, 1))).astype(np.float32)
    _check(matcher, q, t)


def test_l2_exact_duplicates_and_ties(matcher):
    # every query occurs verbatim in the train set (distance exactly 0) and every train row occurs twice
    # (exact ties: best = smaller index, second = its copy)
    rng = np.random.default_rng(22)
    q = rng.standard_normal((513, 128)).astype(np.float32)
    base = np.concatenate([q[rng.permutation(513)], rng.standard_normal((300, 128)).astype(np.float32)])
    t = np.concatenate([base, base])
    bj, bd, sj, sd = _check(matcher, q, t)
    assert (bd == 0).all() and (sd == 0).all() and (sj == bj + len(base)).all()


def test_l2_zero_rows(matcher):
    # all-zero queries and train rows: -d/2 accumulators are exactly 0 for (0, 0) pairs
    rng = np.random.default_rng(23)
    q = rng.standard_normal((200, 64)).astype(np.float32); q[::7] = 0
    t = rng.standard_normal((333, 64)).astype(np.float32); t[5] = 0; t[100] = 0
    _check(matcher, q, t)


@pytest.mark.parametrize("n1,n2,dim", [(300, 500, 128), (1000, 2100, 64), (2600, 1300, 128), (257, 9000, 32)])
def test_l2_both_work_distributions(matcher, n1, n2, dim):
    # the CTA-pair kernel cuts the (row pair, column tile) items into equal segments, one per resident cluster (a
    # segment may cross row pairs: A' reload, candidate slots per segment)
    rng = np.random.default_rng(n1 + n2 + dim)
    q = rng.standard_normal((n1, dim)).astype(np.float32)
    t = rng.standard_normal((n2, dim)).astype(np.float32)
    t[: min(n1, n2) // 2] = q[: min(n1, n2) // 2] + 0.05 * rng.standard_normal((min(n1, n2) // 2, dim)).astype(np.float32)
    _check(matcher, q, t)


def test_l2_underfilled_grid_shape(matcher):
    # 40 row pairs x 8 column tiles: segments of 4-5 items, most of them crossing a row pair
    rng = np.random.default_rng(99)
    q = rng.random((10240, 64), dtype=np.float32)
    t = rng.random((2048, 64), dtype=np.float32)
    _check(matcher, q, t)


# ---- ranking of the CTA-pair kernel (n1 > 128): one fp16 term + certified band + exhaustive fallback --------------
def test_l2_fp16_mode_is_the_default_and_certifies_random_data(matcher):
    rng = np.random.default_rng(31)
    q = rng.random((4096, 128), dtype=np.float32)
    t = rng.random((6000, 128), dtype=np.float32)
    _check(matcher, q, t)
    assert 0 <= matcher.l2_last_fallback_rows() <= 4            # well-spread data: (almost) nothing needs the fallback


def test_l2_fallback_crowded_band(matcher):
    # twelve train rows within 2e-3 of query 7, adjacent (one column group): more than the group's candidate list
    # holds, so the list cannot prove it has the whole band and row 7 is recomputed exhaustively; the answers must
    # still be the oracle's
    rng = np.random.default_rng(32)
    q = rng.standard_normal((600, 128)).astype(np.float32)
    t = rng.standard_normal((3000, 128)).astype(np.float32)
    e = np.zeros(128, dtype=np.float32); e[3] = 1
    for k in range(12):
        t[100 + k] = q[7] + np.float32(0.01 * (12 - k)) * e         # closest copy has the LARGEST index of the twelve
    bj, bd, sj, sd = _check(matcher, q, t)
    assert bj[7] == 111 and sj[7] == 110
    assert matcher.l2_last_fallback_rows() >= 1


def test_l2_fallback_all_identical_train_rows(matcher):
    # every train row is the same vector: every query's band holds the whole train set -> every row takes the
    # fallback; exact ties resolve to the smallest indices
    rng = np.random.default_rng(33)
    q = rng.standard_normal((300, 96)).astype(np.float32)
    t = np.tile(rng.standard_normal((1, 96)).astype(np.float32), (5000, 1))
    bj, bd, sj, sd = _check(matcher, q, t)
    assert (bj == 0).all() and (sj == 1).all()
    assert matcher.l2_last_fallback_rows() == 300


@pytest.mark.parametrize("scale", [1e-18, 3e-6, 1.0, 4e4, 1e15])
def test_l2_fp16_global_scale(matcher, scale):
    # the fp16 operands live under a global power-of-two scale: tiny and huge magnitudes rank like unit ones
    rng = np.random.default_rng(34)
    q = (rng.standard_normal((700, 128)) * scale).astype(np.float32)
    t = (rng.standard_normal((900, 128)) * scale).astype(np.float32)
    bj, bd, sj, sd = matcher.knn2_l2(q, t)
    d = ((q[:, None, :].astype(np.float64) - t[None].astype(np.float64)) ** 2).sum(-1)
    ej = d.argmin(1)
    assert (bj == ej).mean() > 0.99
    np.testing.assert_allclose(bd, d[np.arange(700), bj], rtol=RTOL)
    np.testing.assert_allclose(bd, d.min(1), rtol=RTOL)


def test_l2_wide_dynamic_range_within_rows(matcher):
    # components spanning 2^-30 .. 1 inside every row: the small ones fall below fp16's range under the global scale
    # and only the band's absolute term covers them
    rng = np.random.default_rng(35)
    mag = 2.0 ** rng.uniform(-30, 0, size=(1, 128))
    q = (rng.standard_normal((500, 128)) * mag).astype(np.float32)
    t = (rng.standard_normal((800, 128)) * mag).astype(np.float32)
    _check(matcher, q, t)
