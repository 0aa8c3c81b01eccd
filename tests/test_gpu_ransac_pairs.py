"""Batched fundamental-matrix RANSAC (pgm_ransac_fundamental_pairs_batch_dev) against the numpy oracle.

Scoring, winner, inlier count and mask are float32 in the same operation order on both sides, so they are compared
bit-exactly against oracle/ransac_np.score (re-exported by oracle/ransac_batch_np) applied to the device's own hypotheses (d_hyp_F), and against
pgm_ransac_score on the same F.  The fp64 estimate is compared with the oracle's numpy SVD on the oracle's own samples
(equal F implies equal samples) within a bound set by fp64 rounding, below."""
import ctypes as C

import numpy as np
import pytest

from oracle import ransac_batch_np as R
from photogrammetry_b200 import synthetic
from photogrammetry_b200._lib import PGM_E_INVALID_ARG, PgmatchError

pytestmark = pytest.mark.gpu

# The device and numpy solve the same fp64 least-squares null-vector problem with different backward-stable methods
# (Givens QR + one-sided Jacobi vs LAPACK's SVD).  Both are accurate to ~eps * sigma_1 / (sigma_8 - sigma_9) in the
# null vector, so for a relative singular gap above GAP_MIN = 1e-8 the two fp64 vectors differ by <= ~1e-8 of their
# norm; F = T2^T F0 T1 is then rounded to float32 (relative 6e-8 per entry, one ulp apart at most when the two fp64
# values straddle a rounding boundary).  F_TOL = 1e-6 of max |F| covers both with margin.  Below GAP_MIN the null
# vector is not determined by the data to that accuracy (e.g. duplicated keypoints), so those samples are excluded.
# The sign convention (largest-magnitude component of v positive) is itself decided by rounding when the two largest
# |v_i| are within rounding of each other -- a skew-symmetric F (pure translation) has |v_1| == |v_3| -- so where the
# oracle's relative margin between them is below SIGN_MIN the two F may differ by their sign and are compared up to it.
GAP_MIN = 1e-8
F_TOL = 1e-6
SIGN_MIN = 1e-9


def _assemble(images, matches):
    """images: list of int32[n, 2]; matches: list of (a, b, qi, tj) or ('ref', p, count) = a copy of the first count
    matches of pair p in slots of its own (pairs whose slots overlap would both write the shared mask slots)."""
    offs = np.concatenate([[0], np.cumsum([len(x) for x in images])]).astype(np.int64)
    xy = np.concatenate(images).astype(np.int32)
    pairs, starts, counts, qis, tjs = [], [], [], [], []
    pos = 0
    for m in matches:
        if m[0] == "ref":
            _, p, cnt = m
            a, b, qi, tj = matches[p]
            m = (a, b, qi[:cnt], tj[:cnt])
        a, b, qi, tj = m
        pairs.append((a, b)); starts.append(pos); counts.append(len(qi))
        qis.append(np.asarray(qi, np.int32)); tjs.append(np.asarray(tj, np.int32))
        pos += len(qi)
    qi = np.concatenate(qis) if qis else np.zeros(0, np.int32)
    tj = np.concatenate(tjs) if tjs else np.zeros(0, np.int32)
    return xy, offs, np.array(pairs, np.int32).reshape(-1, 2), qi, tj, np.array(starts, np.int64), np.array(counts, np.int32)


def _two_view_images(seed, n_pairs, per_pair):
    xy, offs, pairs, qi, tj, st, cn = synthetic.two_view_matches(seed, n_pairs, per_pair)
    images = [xy[offs[k]:offs[k + 1]] for k in range(len(offs) - 1)]
    matches = [(int(a), int(b), qi[st[p]:st[p] + cn[p]], tj[st[p]:st[p] + cn[p]]) for p, (a, b) in enumerate(pairs)]
    return images, matches


def _mixed_batch(P=32):
    images, matches = _two_view_images(1, 4, 300)
    n = len(images)
    images.append(np.full((50, 2), (1234, 777), np.int32))            # degenerate: every keypoint the same pixel
    images.append(np.full((50, 2), (1500, 900), np.int32))
    matches.append((n, n + 1, np.arange(50), np.arange(50)[::-1].copy()))
    matches.append(("ref", 0, 0))                                      # count 0
    matches.append(("ref", 1, P - 1))                                  # count P - 1
    matches.append(("ref", 2, P))                                      # count P
    matches.append((0, 0, np.arange(120), np.arange(120)))             # self pair
    return _assemble(images, matches)


def _to_dev(xy, qi, tj):
    import torch
    return (torch.from_numpy(xy).cuda(), torch.from_numpy(np.ascontiguousarray(qi)).cuda(),
            torch.from_numpy(np.ascontiguousarray(tj)).cuda())


def _coords(batch, p):
    xy, offs, pairs, qi, tj, st, cn = batch
    a, b = pairs[p]
    s, c = int(st[p]), int(cn[p])
    return xy[offs[a] + qi[s:s + c].astype(np.int64)], xy[offs[b] + tj[s:s + c].astype(np.int64)]


def _run(matcher, batch, **kw):
    xy, offs, pairs, qi, tj, st, cn = batch
    d_xy, d_qi, d_tj = _to_dev(xy, qi, tj)
    out = matcher.ransac_fundamental_pairs_batch_dev(d_xy, offs, pairs, d_qi, d_tj, st, cn, **kw)
    return tuple(x.cpu().numpy() for x in out)


def _check_scoring(matcher, batch, res, P, thr, rank):
    best, inl, F, mask, hF, hc = res
    st, cn = batch[5], batch[6]
    for p in range(len(cn)):
        s, c = int(st[p]), int(cn[p])
        if c < P:
            assert best[p] == -2 and inl[p] == 0 and not F[p].any() and not mask[s:s + c].any()
            continue
        xy1, xy2 = _coords(batch, p)
        valid = R.rank2(hF[p]) if rank else None
        ec, eb, em = R.score(hF[p], valid, xy1, xy2, thr)
        assert (hc[p] == ec).all(), p
        assert best[p] == eb and inl[p] == em.sum() and (mask[s:s + c] == em).all(), p
        assert (F[p] == (hF[p][eb] if eb >= 0 else 0)).all(), p
        gc, gb, gm = matcher.ransac_score(hF[p], xy1, xy2, thr, None if valid is None else valid.astype(np.uint8))
        assert (gc == hc[p]).all() and gb == best[p] and (gm == mask[s:s + c]).all(), p


def _check_estimate(batch, hF, P, seed, S, skip=()):
    xy, offs, pairs, qi, tj, st, cn = batch
    excluded = total = 0
    for p in range(len(cn)):
        if cn[p] < P or p in skip:
            continue
        a, b = pairs[p]
        xy1, xy2 = _coords(batch, p)
        idx = np.stack([R.sample_indices(int(cn[p]), P, seed, int(a), int(b), s) for s in range(S)])
        Fo, sv = R.estimate(xy1[idx], xy2[idx], return_sv=True)
        gap = (sv[:, 7] - sv[:, 8]) / sv[:, 0]
        keep = gap > GAP_MIN
        scale = np.abs(Fo).reshape(S, 9).max(1)
        err = np.abs(hF[p].astype(np.float64) - Fo).reshape(S, 9).max(1) / scale
        err_flip = np.abs(hF[p].astype(np.float64) + Fo).reshape(S, 9).max(1) / scale
        tied = R.sign_margin(xy1[idx], xy2[idx]) < SIGN_MIN
        err = np.where(tied, np.minimum(err, err_flip), err)
        assert (err[keep] <= F_TOL).all(), (p, err[keep].max())
        excluded += int((~keep).sum()); total += S
    return excluded / max(total, 1)


@pytest.mark.parametrize("rank", [False, True])
def test_scoring_bit_exact_and_estimate(matcher, rank):
    P, S, seed = 32, 300, 5
    batch = _mixed_batch(P)
    for thr in (0.001, 0.0, -0.5):
        res = _run(matcher, batch, n_samples=S, pairs_per_sample=P, threshold=thr, seed=seed, require_rank2=rank,
                   hypotheses=True)
        assert np.isfinite(res[2]).all() and np.isfinite(res[4][:len(batch[6])][batch[6] >= P]).all()
        _check_scoring(matcher, batch, res, P, thr, rank)
    # pair 4 (one pixel repeated) and the self pair 8 (x1 == x2 makes columns of A equal) have no unique null vector
    frac = _check_estimate(batch, res[4], P, seed, S, skip=(4, 8))
    print(f"excluded (relative gap <= {GAP_MIN}): {frac:.4f}")
    assert frac < 0.01


@pytest.mark.parametrize("P", [8, 64])
def test_estimate_other_sample_sizes(matcher, P):
    S, seed = 200, 9
    batch = _assemble(*_two_view_images(3, 3, 200))
    res = _run(matcher, batch, n_samples=S, pairs_per_sample=P, threshold=0.001, seed=seed, require_rank2=False,
               hypotheses=True)
    _check_scoring(matcher, batch, res, P, 0.001, False)
    frac = _check_estimate(batch, res[4], P, seed, S)
    print(f"P={P}: excluded {frac:.4f}")
    assert frac < 0.05


def test_large_pair_and_single_sample(matcher):
    images, matches = _two_view_images(4, 1, 20000)
    batch = _assemble(images, matches)
    for S in (2000, 1):
        res = _run(matcher, batch, n_samples=S, pairs_per_sample=32, threshold=0.001, seed=1, require_rank2=False,
                   hypotheses=True)
        _check_scoring(matcher, batch, res, 32, 0.001, False)
    assert _check_estimate(batch, res[4], 32, 1, 1) == 0.0


def test_self_and_repeated_pairs_identical(matcher):
    images, matches = _two_view_images(6, 2, 150)
    matches = matches + [matches[0], matches[1], matches[0]]          # repeated pairs with copies of the same matches
    batch = _assemble(images, matches)
    best, inl, F, mask = _run(matcher, batch, n_samples=100, pairs_per_sample=32, require_rank2=False)
    st, cn = batch[5], batch[6]
    for p, q in ((0, 2), (1, 3), (0, 4)):
        assert best[p] == best[q] and inl[p] == inl[q] and (F[p] == F[q]).all()
        assert (mask[st[p]:st[p] + cn[p]] == mask[st[q]:st[q] + cn[q]]).all()


def test_pair_sharded_blocks_equal_one_call(matcher):
    images, matches = _two_view_images(7, 16, 120)
    batch = _assemble(images, matches)
    xy, offs, pairs, qi, tj, st, cn = batch
    d_xy, d_qi, d_tj = _to_dev(xy, qi, tj)
    kw = dict(n_samples=150, pairs_per_sample=32, threshold=0.001, seed=3, require_rank2=False)
    ref = [x.cpu().numpy() for x in matcher.ransac_fundamental_pairs_batch_dev(d_xy, offs, pairs, d_qi, d_tj, st, cn, **kw)]
    for ranks in (2, 3, 8):
        blocks = np.array_split(np.arange(len(pairs)), ranks)
        mask = np.zeros_like(ref[3])
        for blk in blocks:
            b, i, F, m = (x.cpu().numpy() for x in matcher.ransac_fundamental_pairs_batch_dev(
                d_xy, offs, pairs[blk], d_qi, d_tj, st[blk], cn[blk], **kw))
            assert (b == ref[0][blk]).all() and (i == ref[1][blk]).all() and (F == ref[2][blk]).all()
            for k, p in enumerate(blk):
                mask[st[p]:st[p] + cn[p]] = m[st[p]:st[p] + cn[p]]
        assert (mask == ref[3]).all()


def _raw_call(matcher, batch, d, sentinel_outputs, **over):
    xy, offs, pairs, qi, tj, st, cn = batch
    d_xy, d_qi, d_tj = d
    best, inl, F, mask = sentinel_outputs
    a = dict(n_images=len(offs) - 1, pairs=pairs, n_pairs=len(pairs), st=st, cn=cn, S=50, P=32, flags=0,
             capacity=int(mask.numel()), xy=d_xy.data_ptr(), qi=d_qi.data_ptr(), best=best.data_ptr())
    a.update(over)
    return matcher._lib.pgm_ransac_fundamental_pairs_batch_dev(
        matcher._h, a["xy"], offs.ctypes.data, a["n_images"], a["pairs"].ctypes.data, a["n_pairs"], a["qi"],
        d_tj.data_ptr(), a["st"].ctypes.data, a["cn"].ctypes.data, a["S"], a["P"], C.c_float(0.001), 0, a["flags"],
        a["best"], inl.data_ptr(), F.data_ptr(), mask.data_ptr(), a["capacity"], None, None)


def test_untouched_slots_refusals_and_host_syncs(matcher):
    import torch
    images, matches = _two_view_images(8, 3, 100)
    batch = _assemble(images, matches)
    xy, offs, pairs, qi, tj, st, cn = batch
    # leave gaps between the pairs' slots: pair p owns [200 p + 10, 200 p + 110) of a 700-slot list
    qi2, tj2 = np.full(700, -7, np.int32), np.full(700, -7, np.int32)
    st2 = np.arange(3, dtype=np.int64) * 200 + 10
    for p in range(3):
        qi2[st2[p]:st2[p] + 100] = qi[st[p]:st[p] + 100]
        tj2[st2[p]:st2[p] + 100] = tj[st[p]:st[p] + 100]
    batch = (xy, offs, pairs, qi2, tj2, st2, cn)
    d = _to_dev(xy, qi2, tj2)
    dev = d[0].device
    outs = (torch.full((3,), -99, dtype=torch.int32, device=dev), torch.full((3,), -99, dtype=torch.int32, device=dev),
            torch.full((3, 3, 3), 7.0, dtype=torch.float32, device=dev), torch.full((700,), 0xAB, dtype=torch.uint8, device=dev))
    bad = [dict(P=7), dict(P=65), dict(S=0), dict(flags=0x8), dict(n_images=-1),
           dict(pairs=np.array([[0, 9], [2, 3], [4, 5]], np.int32)), dict(pairs=np.array([[-1, 1], [2, 3], [4, 5]], np.int32)),
           dict(cn=np.array([100, -1, 100], np.int32)), dict(st=np.array([10, 210, 650], np.int64)),
           dict(st=np.array([-1, 210, 410], np.int64)), dict(capacity=500), dict(xy=None), dict(qi=None), dict(best=None)]
    for over in bad:
        assert _raw_call(matcher, batch, d, outs, **over) == PGM_E_INVALID_ARG, over
        assert _raw_call(matcher, batch, d, outs) == 0                 # a correct call right after a refusal
    torch.cuda.synchronize()
    st_ = matcher.stats()
    assert st_["host_syncs"] == 0 and st_["pairs"] == 3 and st_["kernel_launches"] == 3
    mask = outs[3].cpu().numpy()
    inside = np.zeros(700, bool)
    for p in range(3):
        inside[st2[p]:st2[p] + 100] = True
    assert (mask[~inside] == 0xAB).all() and set(np.unique(mask[inside]).tolist()) <= {0, 1}
    ref = _run(matcher, batch, n_samples=50, pairs_per_sample=32, require_rank2=False)
    assert (outs[0].cpu().numpy() == ref[0]).all() and (mask[inside] == ref[3][inside]).all()
    with pytest.raises(PgmatchError):
        _run(matcher, batch, n_samples=50, pairs_per_sample=4)


def test_non_default_stream(matcher):
    import torch
    batch = _assemble(*_two_view_images(10, 3, 200))
    ref = _run(matcher, batch, n_samples=200, require_rank2=False)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        xy, offs, pairs, qi, tj, st, cn = batch
        d_xy, d_qi, d_tj = _to_dev(xy, qi, tj)
        out = matcher.ransac_fundamental_pairs_batch_dev(d_xy, offs, pairs, d_qi, d_tj, st, cn, n_samples=200,
                                                         require_rank2=False)
        got = [x.cpu().numpy() for x in out]
    for g, r in zip(got, ref):
        assert (g == r).all()


def test_star_sequence_chain(matcher):
    """BASELINE configs[2]: detect + describe -> ratio + cross-check (and the greedy batch with its tail) -> this call on
    all 31 consecutive pairs, at upstream's S = 2000, P = 32, threshold 0.001, rank gate on and off.  Every pair is
    checked as above: counts, winner, inliers, mask and F bit-exact against the oracle's scoring of the device's own
    hypotheses and against pgm_ransac_score, rank decisions against the oracle's rule on the device's F, and F against
    the oracle's fp64 estimate of the oracle's own samples wherever the relative singular gap exceeds GAP_MIN.

    The sequence is one image shifted by 5 px per frame: for the true matches c2 == c1 after the translation-only
    normalisation, so A has equal column pairs and a null space of dimension >= 3.  There the null vector (hence F and
    the rank decision) is not determined by the data, so most samples of the ratio-filtered lists fall under the gap
    rule; the fraction is printed."""
    import torch
    from photogrammetry_b200 import sequence
    from photogrammetry_b200.sharding import consecutive_pairs
    frames = sequence.shifted_frames(sequence.star_gray(), 32, 5).astype(np.float32)
    res = sequence.match_sequence_dev(matcher, torch.from_numpy(frames).cuda(), 50.0, sequence.star_pairs())
    plist = consecutive_pairs(32)
    xy = res.xy.cpu().numpy()
    fo, fstarts, fcounts = matcher.match_ratio_crosscheck_batch_dev(res.desc, res.offsets, plist, 256, 0.8, True, -1)
    S = 2000
    for label, (q, t, starts, counts) in {"ratio": (fo[0], fo[1], fstarts, fcounts),
                                         "greedy+tail": (res.greedy[0], res.greedy[1], res.greedy_starts, res.greedy_counts)}.items():
        batch = (xy, res.offsets, plist, q.cpu().numpy(), t.cpu().numpy(), np.asarray(starts), np.asarray(counts))
        assert (batch[6] >= 32).all(), label
        for rank in (True, False):
            out = matcher.ransac_fundamental_pairs_batch_dev(res.xy, res.offsets, plist, q.contiguous(), t.contiguous(),
                                                             starts, counts, n_samples=S, pairs_per_sample=32,
                                                             threshold=0.001, seed=0, require_rank2=rank, hypotheses=True)
            got = tuple(x.cpu().numpy() for x in out)
            _check_scoring(matcher, batch, got, 32, 0.001, rank)
            if not rank:
                assert (got[0] >= 0).all(), label
        frac = _check_estimate(batch, got[4], 32, 0, S)
        print(f"{label}: samples under the gap rule {frac:.3f}")
