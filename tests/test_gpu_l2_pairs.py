"""Float descriptors, many image pairs per call (pgm_knn2_l2_pairs_batch_dev, pgm_match_l2_ratio_crosscheck_pairs_batch_dev;
run on a B200: -m gpu).

Per pair with n1 > 128 the knn2 batch is bit-identical to the single-pair call (both rank on the certified fp16 path and
compute every reported distance in the same summation order); every pair, n1 <= 128 included, agrees with the oracle
under the tolerance of test_gpu_l2.py.  The ratio + cross-check filter is bit-exact against a numpy float32 filter on the
library's own knn2 batch outputs."""

import numpy as np
import pytest

from oracle import orc
from photogrammetry_b200 import sharding
from photogrammetry_b200._lib import PGM_E_CAPACITY, PGM_E_INVALID_ARG

pytestmark = pytest.mark.gpu
RTOL = 1e-4
SIZES = [0, 1, 2, 127, 128, 129, 255, 256, 257, 1000, 4097]


@pytest.fixture(scope="module")
def torch_dev(matcher):
    import torch
    return torch.device("cuda", matcher.device)


def _images(sizes, dim, seed, scales=None):
    """Image k: a noisy copy of the first rows of one base set (so that near neighbours exist), times scales[k]."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((max(max(sizes), 1), dim)).astype(np.float32)
    imgs = []
    for k, n in enumerate(sizes):
        x = base[rng.permutation(len(base))[:n]] + np.float32(0.05) * rng.standard_normal((n, dim)).astype(np.float32)
        imgs.append((x * np.float32(1.0 if scales is None else scales[k])).astype(np.float32))
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return imgs, np.concatenate(imgs).reshape(-1, dim), offs


def _batch(matcher, torch_dev, all_desc, offs, pairs):
    import torch
    d = torch.from_numpy(all_desc).to(torch_dev)
    bj, bd, sj, sd, starts = matcher.knn2_l2_pairs_batch_dev(d, offs, pairs)
    return [x.cpu().numpy() for x in (bj, bd, sj, sd)], starts


def _rows(res, starts, p, n1):
    return [x[starts[p]:starts[p] + n1] for x in res]


def _assert_oracle(got, q, t, max_ties=0.01):
    """test_gpu_l2.py's tolerance: indices equal except near-ties, distances within 1e-4 relative."""
    exp = orc.l2_knn2(q, t)
    for (gj, gd), (ej, ed) in (((got[0], got[1]), (exp[0], exp[1])), ((got[2], got[3]), (exp[2], exp[3]))):
        assert ((gj >= 0) == (ej >= 0)).all()
        ok = ej >= 0
        np.testing.assert_allclose(gd[ok], ed[ok], rtol=RTOL, atol=1e-6)
        assert (gd[~ok] == -1.0).all()
        rows = np.nonzero(ok & (gj != ej))[0]
        if len(rows):
            dd = ((q[rows].astype(np.float64) - t[gj[rows]].astype(np.float64)) ** 2).sum(-1)
            assert np.allclose(dd, ed[rows], rtol=RTOL, atol=1e-6)
            assert len(rows) <= max(1, max_ties * len(q))


def _assert_bit_identical(got, single):
    for g, s in zip(got, single):
        assert g.dtype == s.dtype and (g.view(np.int32) == s.view(np.int32)).all()


# --- 1 + 2. bit-identity with the single-pair call, agreement with the oracle --------------------------------------------

@pytest.mark.timeout(900)
@pytest.mark.parametrize("dim", [16, 32, 64, 100, 128])
def test_knn2_batch_matches_single_pair_and_oracle(matcher, torch_dev, dim):
    imgs, all_desc, offs = _images(SIZES, dim, seed=dim)
    n = len(SIZES)
    # every ordered pair (both directions, self pairs) and a repeated pair
    pairs = np.array([(a, b) for a in range(n) for b in range(n)] + [(9, 10), (9, 10)], dtype=np.int32)
    res, starts = _batch(matcher, torch_dev, all_desc, offs, pairs)
    assert matcher.stats()["distance_evals"] == sum(len(imgs[a]) * len(imgs[b]) for a, b in pairs)
    for p, (a, b) in enumerate(pairs):
        q, t = imgs[a], imgs[b]
        got = _rows(res, starts, p, len(q))
        if len(q) > 128:
            _assert_bit_identical(got, matcher.knn2_l2(q, t))
        if len(q):
            _assert_oracle(got, q, t)


# --- 3. fallback rows of several pairs in one launch ---------------------------------------------------------------------

def test_knn2_batch_fallback_inside_a_batch(matcher, torch_dev):
    rng = np.random.default_rng(32)
    q_crowd = rng.standard_normal((600, 128)).astype(np.float32)
    t_crowd = rng.standard_normal((3000, 128)).astype(np.float32)
    e = np.zeros(128, dtype=np.float32); e[3] = 1
    for k in range(12):
        t_crowd[100 + k] = q_crowd[7] + np.float32(0.01 * (12 - k)) * e      # test_l2_fallback_crowded_band
    rng = np.random.default_rng(33)
    q_same = rng.standard_normal((300, 128)).astype(np.float32)
    t_same = np.tile(rng.standard_normal((1, 128)).astype(np.float32), (5000, 1))   # test_l2_fallback_all_identical_train_rows
    rng = np.random.default_rng(34)
    q_rand = rng.random((1500, 128), dtype=np.float32)
    t_rand = rng.random((2000, 128), dtype=np.float32)
    imgs = [q_rand, q_crowd, t_crowd, q_same, t_same, t_rand]
    offs = np.concatenate([[0], np.cumsum([len(x) for x in imgs])]).astype(np.int64)
    pairs = np.array([(0, 5), (1, 2), (3, 4), (5, 0)], dtype=np.int32)
    res, starts = _batch(matcher, torch_dev, np.concatenate(imgs), offs, pairs)
    fallback = matcher.l2_last_fallback_rows()
    single_fallback = 0
    for p, (a, b) in enumerate(pairs):
        got = _rows(res, starts, p, len(imgs[a]))
        _assert_bit_identical(got, matcher.knn2_l2(imgs[a], imgs[b]))
        single_fallback += matcher.l2_last_fallback_rows()
        _assert_oracle(got, imgs[a], imgs[b])
    crowd = _rows(res, starts, 1, 600)
    assert crowd[0][7] == 111 and crowd[2][7] == 110
    same = _rows(res, starts, 2, 300)
    assert (same[0] == 0).all() and (same[2] == 1).all()
    # every row of the identical-rows pair and row 7 of the crowded pair, plus the (almost) nothing of well-spread data
    assert 301 <= fallback <= 301 + 8 and 301 <= single_fallback <= 301 + 8


# --- 4. one scale per chunk: images of very different magnitude -----------------------------------------------------------

def test_knn2_batch_images_of_very_different_magnitude(matcher, torch_dev):
    sizes = [700, 600, 800, 500, 900]
    imgs, all_desc, offs = _images(sizes, 96, seed=41, scales=[1.0, 1e-6, 1e6, 1.0, 1e-6])
    pairs = np.array([(0, 1), (1, 2), (2, 3), (3, 0), (1, 4), (4, 1), (2, 2), (0, 3)], dtype=np.int32)
    scales = [1.0, 1e-6, 1e6, 1.0, 1e-6]
    res, starts = _batch(matcher, torch_dev, all_desc, offs, pairs)
    for p, (a, b) in enumerate(pairs):
        got = _rows(res, starts, p, sizes[a])
        _assert_bit_identical(got, matcher.knn2_l2(imgs[a], imgs[b]))
        # across magnitudes every train row is equally far within fp32 resolution (|q|^2 >> the spread of the
        # distances): the indices are near-ties throughout, checked by distance only
        _assert_oracle(got, imgs[a], imgs[b], max_ties=0.01 if scales[a] == scales[b] else 1.0)


# --- 5. chunking -----------------------------------------------------------------------------------------------------------

@pytest.mark.timeout(900)
def test_knn2_batch_chunks(matcher, torch_dev):
    rng = np.random.default_rng(51)
    dim = 32
    small = [130 + (k % 70) for k in range(60)]
    big = [(1 << 20) - 1, 257]
    sizes = small + big
    imgs, all_desc, offs = _images(sizes, dim, seed=52)
    n = len(small)
    pairs = [(int(a), int(b)) for a, b in rng.integers(0, n, size=(5000, 2))]
    pairs += [(n, n + 1)] * 5                         # 5 x 2^20 - 1 query rows: past the row budget of one chunk
    pairs += [(int(a), int(b)) for a, b in rng.integers(0, n, size=(20, 2))]
    pairs = np.array(pairs, dtype=np.int32)
    res, starts = _batch(matcher, torch_dev, all_desc, offs, pairs)
    assert matcher.stats()["kernel_launches"] >= 10     # >= 2 chunks of five kernels
    cache = {}
    for p, (a, b) in enumerate(pairs):
        if (a, b) not in cache:
            cache[(a, b)] = matcher.knn2_l2(imgs[a], imgs[b])
        _assert_bit_identical(_rows(res, starts, p, sizes[a]), cache[(a, b)])


# --- 6. the ratio + cross-check filter -------------------------------------------------------------------------------------

def _ratio_call(matcher, torch_dev, all_desc, offs, pairs, ratio, cross, max_sq, sentinel=True):
    """The C entry point on outputs pre-filled with sentinels."""
    import torch
    d = torch.from_numpy(all_desc).to(torch_dev)
    sizes = np.diff(offs)
    total = int(sizes[pairs[:, 0]].sum())
    qi = torch.full((max(total, 1),), -7, dtype=torch.int32, device=torch_dev)
    tj = torch.full((max(total, 1),), -7, dtype=torch.int32, device=torch_dev)
    dist = torch.full((max(total, 1),), -7.0, dtype=torch.float32, device=torch_dev)
    counts = np.zeros(len(pairs), dtype=np.int32)
    with matcher.torch_ordered(torch_dev):
        matcher._check(matcher._lib.pgm_match_l2_ratio_crosscheck_pairs_batch_dev(
            matcher._h, d.data_ptr(), offs.ctypes.data, len(offs) - 1, pairs.ctypes.data, len(pairs), all_desc.shape[1],
            float(ratio), int(cross), float(max_sq), qi.data_ptr(), tj.data_ptr(), dist.data_ptr(), total, counts.ctypes.data))
    return qi.cpu().numpy(), tj.cpu().numpy(), dist.cpu().numpy(), counts


def _numpy_filter(fwd, rev, n2, ratio, cross, max_sq):
    bj, bd, _, sd = fwd
    rr = np.float32(np.float32(ratio) * np.float32(ratio))
    keep = bj >= 0
    if not (n2 < 2 or np.float32(ratio) <= 0):
        keep &= bd < rr * sd
    if cross:
        i = np.arange(len(bj))
        keep &= np.where(bj >= 0, rev[0][np.clip(bj, 0, None)] if len(rev[0]) else -1, -1) == i
    if max_sq >= 0:
        keep &= bd <= np.float32(max_sq)
    i = np.nonzero(keep)[0].astype(np.int32)
    return i, bj[i], bd[i]


@pytest.mark.timeout(900)
def test_ratio_crosscheck_batch_is_the_filter_of_the_knn2_batch(matcher, torch_dev):
    sizes = [0, 1, 2, 129, 300, 1000, 2500]
    imgs, all_desc, offs = _images(sizes, 128, seed=61)
    pairs = np.array([(4, 5), (5, 4), (6, 5), (3, 3), (5, 1), (1, 5), (2, 6), (4, 0), (0, 4), (6, 6), (4, 5)], dtype=np.int32)
    rev_pairs = pairs[:, ::-1].copy()
    fres, fst = _batch(matcher, torch_dev, all_desc, offs, pairs)
    rres, rst = _batch(matcher, torch_dev, all_desc, offs, rev_pairs)
    for ratio in (0.0, 0.6, 0.8, 1.0):
        for cross in (True, False):
            for max_sq in (-1.0, 20.0):
                qi, tj, dist, counts = _ratio_call(matcher, torch_dev, all_desc, offs, pairs, ratio, cross, max_sq)
                st = matcher.stats()
                evals = sum(sizes[a] * sizes[b] for a, b in pairs)
                assert st["distance_evals"] == evals and st["evals_computed"] == (2 if cross else 1) * evals
                assert st["host_syncs"] <= 2
                start = 0
                for p, (a, b) in enumerate(pairs):
                    n1, n2 = sizes[a], sizes[b]
                    fwd = _rows(fres, fst, p, n1)
                    rev = _rows(rres, rst, p, n2)
                    ei, ej, ed = _numpy_filter(fwd, rev, n2, ratio, cross, max_sq) if n2 else (np.zeros(0, np.int32),) * 3
                    c = counts[p]
                    assert c == len(ei), (ratio, cross, max_sq, p)
                    assert (qi[start:start + c] == ei).all() and (tj[start:start + c] == ej).all()
                    assert (dist[start:start + c].view(np.int32) == np.asarray(ed, np.float32).view(np.int32)).all()
                    assert (np.diff(qi[start:start + c]) > 0).all()
                    assert (qi[start + c:start + n1] == -7).all() and (dist[start + c:start + n1] == -7.0).all()
                    start += n1


def test_ratio_crosscheck_batch_agrees_with_an_oracle_restatement(matcher, torch_dev):
    sizes = [1500, 1400, 1600, 900]
    imgs, all_desc, offs = _images(sizes, 128, seed=71)
    pairs = np.array([(a, b) for a in range(4) for b in range(4) if a != b], dtype=np.int32)
    qi, tj, dist, counts = _ratio_call(matcher, torch_dev, all_desc, offs, pairs, 0.8, True, -1.0)
    start = 0
    for p, (a, b) in enumerate(pairs):
        q, t = imgs[a], imgs[b]
        fwd, rev = orc.l2_knn2(q, t), orc.l2_knn2(t, q)
        ei, ej, _ = _numpy_filter(fwd, rev, len(t), 0.8, True, -1.0)
        got = set(zip(qi[start:start + counts[p]].tolist(), tj[start:start + counts[p]].tolist()))
        exp = set(zip(ei.tolist(), ej.tolist()))
        for i, j in got ^ exp:
            # a documented near-tie: the row's ratio sits at the threshold, or a best neighbour in either direction is
            # tied with another within the distance tolerance
            b1, b2 = fwd[1][i], fwd[3][i]
            at_ratio = abs(b1 - np.float32(0.64) * b2) <= RTOL * max(b1, 1e-6)
            tie_fwd = fwd[3][i] <= fwd[1][i] * (1 + RTOL) + 1e-6
            jj = fwd[0][i]
            tie_rev = rev[3][jj] <= rev[1][jj] * (1 + RTOL) + 1e-6
            assert at_ratio or tie_fwd or tie_rev, (p, i, j)
        assert len(got ^ exp) <= 0.01 * len(q)
        start += len(q)


# --- 7. refusals -----------------------------------------------------------------------------------------------------------

def test_refusals_then_correct_calls(matcher, torch_dev):
    import torch
    rng = np.random.default_rng(81)
    q = rng.standard_normal((300, 64)).astype(np.float32)
    t = rng.standard_normal((400, 64)).astype(np.float32)
    before = matcher.knn2_l2(q, t)
    all_desc = np.concatenate([q, t])
    d = torch.from_numpy(all_desc).to(torch_dev)
    offs = np.array([0, 300, 700], dtype=np.int64)
    pairs = np.array([(0, 1), (1, 0)], dtype=np.int32)
    out = [torch.empty(700, dtype=dt, device=torch_dev) for dt in (torch.int32, torch.float32, torch.int32, torch.float32)]
    lib, h = matcher._lib, matcher._h

    def knn(dim=64, pl=pairs, of=offs, cap=700, ptr=d.data_ptr(), outs=out):
        return lib.pgm_knn2_l2_pairs_batch_dev(h, ptr, of.ctypes.data, len(of) - 1, pl.ctypes.data, len(pl), dim,
                                               *(o.data_ptr() if o is not None else None for o in outs), cap)

    def ratio(dim=64, pl=pairs, cap=700, ptr=d.data_ptr()):
        counts = np.zeros(len(pl), dtype=np.int32)
        return lib.pgm_match_l2_ratio_crosscheck_pairs_batch_dev(
            h, ptr, offs.ctypes.data, 2, pl.ctypes.data, len(pl), dim, 0.8, 1, -1.0, out[0].data_ptr(), out[2].data_ptr(),
            out[1].data_ptr(), cap, counts.ctypes.data)

    huge = np.array([0, 300, 300 + (1 << 20)], dtype=np.int64)
    bad_pairs = np.array([(0, 2)], dtype=np.int32)
    neg_pairs = np.array([(-1, 0)], dtype=np.int32)
    for fn in (knn, ratio):
        assert fn(dim=0) == PGM_E_INVALID_ARG
        assert fn(dim=129) == PGM_E_INVALID_ARG
        assert fn(pl=bad_pairs) == PGM_E_INVALID_ARG
        assert fn(pl=neg_pairs) == PGM_E_INVALID_ARG
        assert fn(cap=699) == PGM_E_CAPACITY
        assert fn(ptr=None) == PGM_E_INVALID_ARG
    assert knn(of=huge) == PGM_E_INVALID_ARG
    assert knn(outs=[out[0], None, out[2], out[3]]) == PGM_E_INVALID_ARG
    assert knn() == 0
    torch.cuda.synchronize(torch_dev)
    _assert_bit_identical([x.cpu().numpy()[:300] for x in out], matcher.knn2_l2(q, t))
    _assert_bit_identical([x.cpu().numpy()[300:] for x in out], matcher.knn2_l2(t, q))
    _assert_bit_identical(matcher.knn2_l2(q, t), before)


# --- 8. streams, sharding, stats --------------------------------------------------------------------------------------------

def test_stream_sharding_and_stats(matcher, torch_dev):
    import torch
    sizes = [300, 1000, 0, 129, 700, 2000]
    imgs, all_desc, offs = _images(sizes, 128, seed=91)
    pairs = np.array([(a, b) for a in range(6) for b in range(6) if a != b], dtype=np.int32)
    ref, starts = _batch(matcher, torch_dev, all_desc, offs, pairs)
    st = matcher.stats()
    evals = sum(sizes[a] * sizes[b] for a, b in pairs)
    assert st["distance_evals"] == evals and st["evals_computed"] == evals and st["host_syncs"] <= 2
    d = torch.from_numpy(all_desc).to(torch_dev)
    s = torch.cuda.Stream(torch_dev)
    with torch.cuda.stream(s):
        got = matcher.knn2_l2_pairs_batch_dev(d, offs, pairs)
        got = [x.cpu().numpy() for x in got[:4]]
    _assert_bit_identical(got, ref)
    full = _triples(_ratio_call(matcher, torch_dev, all_desc, offs, pairs, 0.8, True, -1.0), offs, pairs)
    for world in (2, 3, 8):
        blocks = [_triples(_ratio_call(matcher, torch_dev, all_desc, offs, pairs[lo:hi], 0.8, True, -1.0), offs, pairs[lo:hi])
                  for lo, hi in sharding.partition_pairs(pairs, sizes, world) if hi > lo]
        got = [t for b in blocks for t in b]
        assert len(got) == len(full)
        for g, f in zip(got, full):
            assert all((x == y).all() for x, y in zip(g, f))


def _triples(call, offs, pairs):
    """Per pair: (qi, tj, dist) of one ratio call."""
    qi, tj, dist, counts = call
    starts = np.concatenate([[0], np.cumsum(np.diff(offs)[pairs[:, 0]])]).astype(np.int64)
    return [(qi[o:o + c], tj[o:o + c], dist[o:o + c].view(np.int32)) for o, c in zip(starts, counts)]
