"""The numpy oracle of the batched fundamental-matrix RANSAC (oracle/ransac_batch_np.py): its sampler, its fp64 8-point
estimate and its sign convention.  CPU only."""
import numpy as np
from scipy import stats

from oracle import ransac_batch_np as R


def test_sampler_distinct_in_range_and_deterministic():
    for count, P in [(8, 8), (9, 8), (32, 32), (33, 32), (100, 64), (20000, 32), (2**31 - 1, 64)]:
        for s in range(20):
            idx = R.sample_indices(count, P, 7, 3, 5, s)
            assert len(idx) == P and len(set(idx.tolist())) == P
            assert idx.min() >= 0 and idx.max() < count and (np.diff(idx) > 0).all()
            assert (idx == R.sample_indices(count, P, 7, 3, 5, s)).all()
    # the key depends on seed, pair and sample
    base = R.sample_indices(1000, 32, 7, 3, 5, 0)
    for other in [(8, 3, 5, 0), (7, 4, 5, 0), (7, 3, 6, 0), (7, 3, 5, 1), (7, 5, 3, 0)]:
        assert (R.sample_indices(1000, 32, *other) != base).any()


def test_sampler_is_uniform():
    # every index of [0, count) is drawn with probability P / count: chi^2 over 4000 samples of 8 out of 50
    count, P, n = 50, 8, 4000
    hits = np.zeros(count)
    for s in range(n):
        hits[R.sample_indices(count, P, 11, 0, 1, s)] += 1
    chi2 = ((hits - n * P / count) ** 2 / (n * P / count)).sum()
    assert stats.chi2.sf(chi2, count - 1) > 1e-3, chi2
    # and every subset size-1 marginal of the first and last positions is uniform too (Floyd's draws are unbiased)
    firsts = np.array([R.sample_indices(count, P, 11, 0, 1, s)[0] for s in range(n)])
    assert firsts.max() <= count - P


def _epipolar_points(F, n, rng):
    """float (x1, x2) with x2^T F x1 == 0 up to rounding: x2 on the epipolar line F x1."""
    x1 = rng.uniform(0, 4000, (n, 2))
    h1 = np.concatenate([x1, np.ones((n, 1))], 1)
    line = h1 @ F.T                                       # l = F x1
    u = rng.uniform(0, 4000, n)
    v = -(line[:, 0] * u + line[:, 2]) / line[:, 1]
    return x1, np.stack([u, v], 1)


def test_estimate_annihilates_noise_free_correspondences():
    rng = np.random.default_rng(3)
    U, _, Vt = np.linalg.svd(rng.standard_normal((3, 3)))
    Ftrue = U @ np.diag([1.0, 0.3, 0.0]) @ Vt             # rank 2
    for P in (8, 32, 64):
        x1, x2 = _epipolar_points(Ftrue, P, rng)
        F, sv = R.estimate(x1, x2, return_sv=True)
        F = F.astype(np.float64)
        # the estimate satisfies x2^T F x1 = 0 (the form A v = c2^T F0 c1 annihilates), to the float32 rounding of A.
        # It is not compared with Ftrue entry by entry: without upstream's scaling step (Pow(x, 0) == 1) the columns of
        # A differ in scale by ~4e6 and the relative gap sigma_8 / sigma_1 is ~5e-6, so the float32 rows of A leave the
        # entries that multiply the small columns poorly determined -- by the reference's own construction.
        h1 = np.concatenate([x1, np.ones((P, 1))], 1)
        h2 = np.concatenate([x2, np.ones((P, 1))], 1)
        res = np.einsum("ni,ij,nj->n", h2, F, h1)
        scale = np.abs(h2).max() * np.abs(F).max() * np.abs(h1).max()
        assert np.abs(res).max() <= 1e-7 * scale, (P, np.abs(res).max() / scale)
        assert sv[8] <= 1e-12 * sv[0] and sv[7] > 1e-8 * sv[0]       # a one-dimensional null space, found


def test_sign_convention():
    rng = np.random.default_rng(4)
    x1 = rng.integers(0, 4000, (40, 32, 2))
    x2 = x1 + rng.integers(-30, 31, (40, 32, 2))
    A, T1, T2 = R.design_matrix(x1, x2)
    _, _, vh = np.linalg.svd(A.astype(np.float64))
    F = R.estimate(x1, x2).astype(np.float64)
    # recover v from F = T2^T F0 T1 and check that its largest-magnitude component is positive
    F0 = np.linalg.inv(np.swapaxes(T2, -1, -2)) @ F @ np.linalg.inv(T1)
    v = np.swapaxes(F0, -1, -2).reshape(-1, 9)
    k = np.argmax(np.abs(v), axis=1)
    assert (v[np.arange(len(v)), k] > 0).all()
    assert np.allclose(np.abs(v), np.abs(vh[:, -1, :]), atol=1e-4)
    # ties: the lowest index wins, so (-1, 1, 0, ...) / sqrt 2 flips to (1, -1, ...)
    tie = np.zeros(9)
    tie[0], tie[1] = -1.0, 1.0
    assert np.argmax(np.abs(tie)) == 0


def test_rank_gate():
    F = np.diag([1.0, 0.5, 0.0]).astype(np.float32)
    assert R.rank2(F)
    assert not R.rank2(np.diag([1.0, 0.5, 1e-3]).astype(np.float32))
    assert not R.rank2(np.diag([1.0, 0.0, 0.0]).astype(np.float32))
    # 3 ulp_f32(sigma_0) is the boundary: 2^-23 * 3 at sigma_0 = 1 is still "zero", 2^-20 is not
    assert R.rank2(np.diag([1.0, 0.5, 3 * 2.0 ** -23]).astype(np.float32))
    assert not R.rank2(np.diag([1.0, 0.5, 2.0 ** -20]).astype(np.float32))


def test_get_fundamental_pairs_layout():
    from photogrammetry_b200 import synthetic
    xy, offs, pairs, qi, tj, starts, counts = synthetic.two_view_matches(5, 3, 40)
    counts = counts.copy()
    counts[1] = 31                                        # below P: -2
    res = R.get_fundamental_pairs(xy, offs, pairs, qi, tj, starts, counts, 30, 32, 0.001, 0, require_rank2=False)
    assert res[1][0] == -2 and res[1][1] == 0 and not res[1][2].any()
    for best, inl, F, mask, hF, hc in (res[0], res[2]):
        assert hF.shape == (30, 3, 3) and hc.shape == (30,) and best == int(np.argmax(hc))
        assert inl == mask.sum() == hc[best] and (F == hF[best]).all()
