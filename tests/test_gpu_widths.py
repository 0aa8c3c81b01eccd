"""Every descriptor width the C ABI accepts, at shapes that reach each engine (run on a B200: -m gpu).

Rows of 16, 32, 48 and 64 bytes select the 4-, 8-, 12- and 16-word instantiation of every Hamming kernel (round,
tail, finisher, knn2, sorted rows, ratio / cross-check batch), and each width has its own popcount form
(pgm_kernels.cuh, hamming_words / hamming_words_deep).  Every comparison with the oracle is bit-exact, as in
test_gpu_parity.py; the oracle takes the row stride, so the same reference serves every width."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import detect_np as D
from oracle import orc
from photogrammetry_b200 import sharding, synthetic
from photogrammetry_b200._lib import PGM_E_INVALID_ARG, PGM_FLAG_REFERENCE_COMPAT_TAIL, PgmatchError, pinned_empty
from photogrammetry_b200.descriptors import pack_descriptors

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# (desc_bits, stride_bytes): every row width, a partial last word at each, and 256 bits in rows wider than needed
WIDTHS = [(64, 16), (128, 16), (200, 32), (300, 48), (384, 48), (512, 64), (256, 64)]
WIDE = [(128, 16), (384, 48), (512, 64)]
RATIO_GRID = [(0.8, True, -1), (0.9, False, -1), (0.0, True, -1), (0.0, False, 75), (0.7, True, 60)]


def _wid(w):
    return f"{w[0]}b{w[1]}B"


def _assert_clean(a, bits):
    """No bit at position >= bits is set (descriptors are little-endian integers): a mismatch is then the engine's."""
    high = np.packbits((np.arange(a.shape[1] * 8) >= bits).astype(np.uint8), bitorder="little")
    assert not (a & high).any(), "descriptor generator set bits above desc_bits"


def _uniform(seed, n, bits, stride):
    a = synthetic.uniform_descriptors(seed, n, bits, stride)
    assert a.shape == (n, stride)
    _assert_clean(a, bits)
    return a


def _noisy(seed, q, bits):
    a = synthetic.noisy_copy_descriptors(seed, q, bits)
    _assert_clean(a, bits)
    return a


def _pair(seed, n1, n2, dist, bits, stride):
    """U: independent uniform sets; C: the train set is a noisy copy of the queries (near matches and outliers)."""
    if dist == "U":
        return _uniform(seed, n1, bits, stride), _uniform(seed + 1, n2, bits, stride)
    q = _uniform(seed, max(n1, n2), bits, stride)
    return q[:n1], _noisy(seed + 1, q, bits)[:n2]


def _widen(a, stride):
    out = np.zeros((a.shape[0], stride), dtype=np.uint8)
    out[:, :a.shape[1]] = a
    return out


def _expect(got, exp, tail, n1, n2):
    exp = exp if tail else exp[:min(n1, n2)]
    assert got.shape == exp.shape and (got == exp).all()


# --- 1. single pair, latency mode ---------------------------------------------------------------------------------

@pytest.mark.parametrize("n1,n2,dist,tail", [(3000, 2800, "U", True), (2048, 2048, "C", True),
                                             (2500, 1800, "U", True), (2500, 1800, "U", False),
                                             (1800, 2500, "C", True), (1800, 2500, "C", False)])
@pytest.mark.parametrize("bits,stride", WIDTHS, ids=[_wid(w) for w in WIDTHS])
def test_greedy_latency_mode_per_width(matcher, bits, stride, n1, n2, dist, tail):
    q, t = _pair(bits * 7 + n1, n1, n2, dist, bits, stride)
    exp = orc.match_sweep(q, t)
    got = matcher.match_greedy(q, t, bits, reference_compat_tail=tail)
    _expect(got, exp, tail, n1, n2)
    assert matcher.stats()["distance_evals"] == n1 * n2


@pytest.mark.parametrize("dist", ["U", "C"])
@pytest.mark.parametrize("bits,stride", [(384, 48), (512, 64), (256, 64)], ids=["384b48B", "512b64B", "256b64B"])
def test_greedy_8k_per_width(matcher, bits, stride, dist):
    # large enough for the round kernel's large tiles and the candidate-edge passes
    q, t = _pair(bits + 3, 8192, 8192, dist, bits, stride)
    exp = orc.match_sweep(q, t)
    got = matcher.match_greedy(q, t, bits)
    assert (got == exp).all()
    st = matcher.stats()
    assert st["distance_evals"] == 8192 * 8192
    if dist == "U":
        # the bound test_gpu_parity.py holds at 256 bits: a candidate-edge path that silently stopped pruning at this
        # width would still be correct, but would recompute every distance in every pass
        assert st["evals_computed"] < 2.5 * st["distance_evals"]


def test_greedy_distance_512_edges(matcher, monkeypatch):
    # 64-byte rows are the only ones with a distance of 512 (a row and its complement).  1000 other queries can take at
    # most 1000 of the 1400 complement rows, so at least 400 matches are made at that distance, with the sparse phase's
    # edge list both at full and at the smallest capacity
    bits, stride = 512, 64
    a = _uniform(91, 1, bits, stride)
    q = np.concatenate([np.repeat(a, 1500, axis=0), _uniform(92, 1000, bits, stride)])
    t = np.concatenate([np.repeat(~a, 1400, axis=0), _uniform(93, 800, bits, stride)])
    rng = np.random.default_rng(94)
    q, t = q[rng.permutation(len(q))], t[rng.permutation(len(t))]
    assert orc.hamming(a, ~a) == 512
    exp = orc.match_sweep(q, t)
    assert (exp[:len(t), 2] == 512).any()
    assert (matcher.match_greedy(q, t, bits) == exp).all()
    monkeypatch.setenv("PGM_SP_SLOTS_MAX", "1")
    assert (matcher.match_greedy(q, t, bits) == exp).all()


# --- 2. sparse-phase truncation, candidate-list overflow, heavy ties ----------------------------------------------

def _batch17(matcher, q, t, bits):
    """The same pair 17 times: more than 16 pairs, so the throughput engine (standalone kernels) runs."""
    imgs = np.concatenate([q, t])
    offs = np.array([0, len(q), len(q) + len(t)], dtype=np.int64)
    tr, starts, counts = matcher.match_pairs_batch(imgs, offs, np.array([(0, 1)] * 17, dtype=np.int32), bits)
    return [tr[starts[p]:starts[p] + counts[p]] for p in (0, 16)]


@pytest.mark.parametrize("slots_max", [1, 5])
@pytest.mark.parametrize("n1,n2,dist", [(3000, 2800, "U"), (2048, 2048, "C"), (4096, 4096, "U")])
@pytest.mark.parametrize("bits,stride", WIDE, ids=[_wid(w) for w in WIDE])
def test_sparse_phase_truncated_edge_list_per_width(matcher, monkeypatch, bits, stride, n1, n2, dist, slots_max):
    q, t = _pair(1234 + bits, n1, n2, dist, bits, stride)
    exp = orc.match_sweep(q, t)
    monkeypatch.setenv("PGM_SP_SLOTS_MAX", str(slots_max))
    got = matcher.match_greedy(q, t, bits)
    assert got.shape == exp.shape and (got == exp).all()
    for g in _batch17(matcher, q, t, bits):
        assert (g == exp).all()


def _bimodal(seed, n, bits, stride, dup_frac=0.5):
    """Half the rows are copies of one descriptor, the rest uniform: the duplicate block alone lists ~n^2/4 edges, far
    more than any candidate list holds (as in test_gpu_parity.py, at this width)."""
    a = _uniform(seed, n, bits, stride)
    a[:int(n * dup_frac)] = a[0]
    return a[np.random.default_rng(seed).permutation(n)]


@pytest.mark.parametrize("n1,n2", [(3000, 3000), (2500, 1800), (700, 900)])
@pytest.mark.parametrize("bits,stride", WIDE, ids=[_wid(w) for w in WIDE])
def test_candidate_list_overflow_per_width(matcher, bits, stride, n1, n2):
    q, t = _bimodal(5, n1, bits, stride), _bimodal(6, n2, bits, stride)
    t[: n2 // 2] = q[0]
    exp = orc.match_sweep(q, t)
    assert (matcher.match_greedy(q, t, bits) == exp).all()
    imgs = np.concatenate([q[:600], t[:600]] + [_bimodal(20 + k, 600, bits, stride) for k in range(5)])
    offs = np.arange(8, dtype=np.int64) * 600
    pairs = sharding.all_pairs(7)
    tr, starts, counts = matcher.match_pairs_batch(imgs, offs, pairs, bits)
    for p in (0, 1, 7, 20):
        a, b = pairs[p]
        e = orc.match_sweep(imgs[offs[a]:offs[a + 1]], imgs[offs[b]:offs[b + 1]])
        assert (tr[starts[p]:starts[p] + counts[p]] == e).all(), p
    outs, _ = sharding.match_train_sharded_emulated(matcher, q, t, 3, desc_bits=bits)
    assert all((o == exp).all() for o in outs)


@pytest.mark.parametrize("slots_max", [None, 1])
@pytest.mark.parametrize("bits", [32, 64])
def test_heavy_ties_3000(matcher, monkeypatch, bits, slots_max):
    # 33 or 65 distinct distances: every stage's (distance, index) tie-break decides most matches
    q, t = _pair(bits, 3000, 3000, "U", bits, 16)
    t[100:400] = _noisy(bits + 9, q[:300], bits)
    exp = orc.match_sweep(q, t)
    if slots_max:
        monkeypatch.setenv("PGM_SP_SLOTS_MAX", str(slots_max))
    assert (matcher.match_greedy(q, t, bits) == exp).all()
    for g in _batch17(matcher, q, t, bits):
        assert (g == exp).all()
    for a, b in zip(matcher.knn2(q, t, bits), orc.knn2(q, t)):
        assert (a == b).all()


# --- 3. the batch engine ------------------------------------------------------------------------------------------

SIZES = [0, 1, 17, 300, 2500, 1200, 700, 64, 2048, 999, 1500, 5, 2200, 128, 513, 1800, 40, 2400, 900, 260]
PAIRS = [(4, 8), (8, 4), (3, 5), (5, 3), (12, 17), (17, 12), (0, 4), (1, 2), (2, 1), (6, 9), (9, 6), (10, 15),
         (15, 10), (13, 14), (14, 13), (7, 16), (16, 7), (11, 19), (19, 18), (18, 19), (3, 3), (4, 17), (17, 4),
         (8, 8), (2, 11), (11, 2)]


def _images(bits, stride):
    imgs = [_uniform(300 + 11 * k + bits, n, bits, stride) for k, n in enumerate(SIZES)]
    imgs[8] = _noisy(bits + 1, imgs[4][:2048], bits)              # near matches between images 4 and 8
    imgs[17][:1000] = _noisy(bits + 2, imgs[12][:1000], bits)
    imgs[5][:40] = imgs[5][0]                                      # duplicate rows
    offs = np.concatenate([[0], np.cumsum(SIZES)]).astype(np.int64)
    return imgs, np.concatenate(imgs), offs


_sweeps = {}


def _sweep(bits, stride, imgs, a, b):
    key = (bits, stride, a, b)
    if key not in _sweeps:
        _sweeps[key] = orc.match_sweep(imgs[a], imgs[b])
    return _sweeps[key]


def _check_batch(imgs, bits, stride, pairs, tr, starts, counts, tail):
    for p, (a, b) in enumerate(pairs):
        n1, n2 = len(imgs[a]), len(imgs[b])
        assert counts[p] == (n1 if tail else min(n1, n2)), p
        exp = _sweep(bits, stride, imgs, a, b)
        got = tr[starts[p]:starts[p] + counts[p]]
        assert (got == exp[:counts[p]]).all(), (p, a, b)
        # without the tail, the header promises -1 in every unused slot of the pair's range
        assert (tr[starts[p] + counts[p]:starts[p] + n1] == -1).all(), (p, a, b)


@pytest.mark.parametrize("tail", [True, False])
@pytest.mark.parametrize("mode", ["latency", "throughput"])
@pytest.mark.parametrize("bits,stride", WIDTHS, ids=[_wid(w) for w in WIDTHS])
def test_batch_per_width(matcher, bits, stride, mode, tail):
    import torch
    imgs, all_desc, offs = _images(bits, stride)
    pairs = np.array(PAIRS[:12] if mode == "latency" else PAIRS, dtype=np.int32)      # <= 16 pairs: latency mode
    n1s = np.array([SIZES[a] for a, _ in pairs])
    starts = np.concatenate([[0], np.cumsum(n1s)[:-1]])
    total = int(n1s.sum())
    tr, st, counts = matcher.match_pairs_batch(all_desc, offs, pairs, bits, reference_compat_tail=tail)
    assert (st == starts).all()
    _check_batch(imgs, bits, stride, pairs, tr, starts, counts, tail)
    # the device-pointer form, outputs pre-filled with garbage
    dev = torch.device("cuda", matcher.device)
    d_all = torch.from_numpy(all_desc).to(dev)
    out = torch.full((3, total), 12345, dtype=torch.int32, device=dev)
    with matcher.torch_ordered():
        dcounts = matcher.match_pairs_batch_dev(d_all.data_ptr(), offs, pairs, bits, stride, out[0].data_ptr(),
                                                out[1].data_ptr(), out[2].data_ptr(), total, reference_compat_tail=tail)
    torch.cuda.synchronize()
    assert (dcounts == counts).all()
    _check_batch(imgs, bits, stride, pairs, out.T.cpu().numpy(), starts, dcounts, tail)


def test_batch_many_chunks_pinned_outputs_512(matcher):
    # more than 4096 pairs (two chunks and part of a third) at 16 words, written straight into page-locked arrays
    bits, stride = 512, 64
    n_img, per = 150, 24
    imgs = [_uniform(700 + k, per, bits, stride) for k in range(n_img)]
    for k in range(1, n_img, 3):
        imgs[k][:12] = _noisy(k, imgs[k - 1], bits)[:12]
    all_desc = np.concatenate(imgs)
    offs = np.arange(n_img + 1, dtype=np.int64) * per
    pairs = np.array([(a, b) for a in range(n_img) for b in range(a + 1, n_img)], dtype=np.int32)
    total = len(pairs) * per
    for tail in (True, False):
        out = pinned_empty((3, total), np.int32)
        out[:] = -7
        got, starts, counts = matcher.match_pairs_batch(all_desc, offs, pairs, bits, reference_compat_tail=tail, out=out)
        assert (counts == per).all()
        for p in list(range(0, len(pairs), 331)) + [4095, 4096, 8191, 8192, len(pairs) - 1]:
            a, b = pairs[p]
            assert (got[:, starts[p]:starts[p] + per].T == orc.match_sweep(imgs[a], imgs[b])).all(), p
        assert (np.sort(got[0].reshape(len(pairs), per), axis=1) == np.arange(per)).all()


# --- 4. a wider row than the width needs changes nothing ----------------------------------------------------------

@pytest.mark.parametrize("bits,narrow,wide", [(256, 32, 64), (128, 16, 48)])
def test_wider_stride_changes_nothing(matcher, bits, narrow, wide):
    q = _uniform(bits + 17, 3000, bits, narrow)
    t = _noisy(bits + 18, q, bits)[:2600]
    qw, tw = _widen(q, wide), _widen(t, wide)
    exp = orc.match_sweep(q, t)
    for tail in (True, False):
        a = matcher.match_greedy(q, t, bits, reference_compat_tail=tail)
        _expect(a, exp, tail, 3000, 2600)
        assert (matcher.match_greedy(qw, tw, bits, reference_compat_tail=tail) == a).all()
    imgs, all_desc, offs = _images(bits, narrow)
    pairs = np.array(PAIRS, dtype=np.int32)
    for tail in (True, False):
        narrow_out = matcher.match_pairs_batch(all_desc, offs, pairs, bits, reference_compat_tail=tail)
        wide_out = matcher.match_pairs_batch(_widen(all_desc, wide), offs, pairs, bits, reference_compat_tail=tail)
        assert all((x == y).all() for x, y in zip(narrow_out, wide_out))
    for x, y, z in zip(matcher.knn2(q, t, bits), matcher.knn2(qw, tw, bits), orc.knn2(q, t)):
        assert (x == y).all() and (x == z).all()
    for ratio, cc, md in RATIO_GRID:
        x = matcher.match_ratio_crosscheck(q, t, ratio, cc, md, bits)
        assert (x == matcher.match_ratio_crosscheck(qw, tw, ratio, cc, md, bits)).all(), (ratio, cc, md)
    x = matcher.match_keypoints_sorted(q[:200], t, bits)
    assert (x == matcher.match_keypoints_sorted(qw[:200], tw, bits)).all()
    assert (x == orc.python_twin(q[:200], t)).all()


# --- 5. knn2, ratio / cross-check, sorted rows --------------------------------------------------------------------

@pytest.mark.parametrize("n1,n2", [(3000, 20000), (20000, 3000)])
@pytest.mark.parametrize("bits,stride", WIDTHS, ids=[_wid(w) for w in WIDTHS])
def test_knn2_per_width(matcher, bits, stride, n1, n2):
    q = _uniform(bits + 40, n1, bits, stride)
    t = _uniform(bits + 41, n2, bits, stride)
    m = min(n1, n2) // 2
    t[:m] = _noisy(bits + 42, q[:m], bits)
    t[7:11] = t[7]                                      # duplicate train rows: ties on the column splits
    for a, b in zip(matcher.knn2(q, t, bits), orc.knn2(q, t)):
        assert a.shape == b.shape and (a == b).all()


@pytest.mark.parametrize("bits,stride", WIDTHS, ids=[_wid(w) for w in WIDTHS])
def test_ratio_crosscheck_and_sorted_rows_per_width(matcher, bits, stride):
    q = _uniform(bits + 50, 3000, bits, stride)
    t = _noisy(bits + 51, q, bits)[:2500]
    for ratio, cc, md in RATIO_GRID:
        got = matcher.match_ratio_crosscheck(q, t, ratio, cc, md, bits)
        exp = orc.match_ratio_crosscheck(q, t, ratio, cc, md)
        assert got.shape == exp.shape and (got == exp).all(), (ratio, cc, md)
    ts = _uniform(bits + 52, 3000, bits, stride)
    ts[:100] = _noisy(bits + 53, q[:100], bits)
    got = matcher.match_keypoints_sorted(q[:200], ts, bits)
    assert (got == orc.python_twin(q[:200], ts)).all()
    # the batched kernel (one CTA per pair, both sets in shared memory) on slices of the same pair, both directions
    import torch
    imgs = [q[:600], t[:500], q[600:1000], t[500:1300], q[1000:1001]]
    offs = np.concatenate([[0], np.cumsum([len(x) for x in imgs])]).astype(np.int64)
    pairs = np.array([(0, 1), (1, 0), (2, 3), (3, 2), (4, 3), (3, 4), (2, 2)], dtype=np.int32)
    d_all = torch.from_numpy(np.concatenate(imgs)).cuda()
    for ratio, cc, md in RATIO_GRID:
        out, starts, counts = matcher.match_ratio_crosscheck_batch_dev(d_all, offs, pairs, bits, ratio, cc, md)
        out = out.cpu().numpy()
        for p, (a, b) in enumerate(pairs):
            exp = orc.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md)
            got = out[:, starts[p]:starts[p] + counts[p]].T
            assert got.shape == exp.shape and (got == exp).all(), (ratio, cc, md, p)


# --- 6. the batched ratio / cross-check kernel at its shared-memory bound -----------------------------------------

RCB_SMEM_MAX = 200 * 1024


@pytest.mark.parametrize("bits,stride,n1,n2", [(128, 16, 6549, 5000), (384, 48, 2637, 1504), (512, 64, 1606, 1500)])
def test_ratio_crosscheck_batch_at_shared_memory_bound(matcher, bits, stride, n1, n2):
    import torch
    # both descriptor sets and the column minima in one CTA: (n1 + n2) * stride + 4 * n2 + 16 <= 200 KB (include/pgmatch.h)
    assert (n1 + n2) * stride + 4 * n2 + 16 == RCB_SMEM_MAX
    q = _uniform(bits + 60, n1 + 1, bits, stride)
    t = _noisy(bits + 61, q, bits)[:n2 + 1]
    d_all = torch.from_numpy(np.concatenate([q, t])).cuda()
    # images: 0 = q[:n1], 1 = q[n1], 2 = t[:n2], 3 = t[n2]
    offs = np.array([0, n1, n1 + 1, n1 + 1 + n2, n1 + 2 + n2], dtype=np.int64)
    pairs = np.array([(0, 2), (1, 3), (1, 2), (3, 1)], dtype=np.int32)
    imgs = [q[:n1], q[n1:], t[:n2], t[n2:]]
    for ratio, cc, md in [(0.8, True, -1), (0.0, False, -1), (0.7, True, bits // 4)]:
        out, starts, counts = matcher.match_ratio_crosscheck_batch_dev(d_all, offs, pairs, bits, ratio, cc, md)
        out = out.cpu().numpy()
        for p, (a, b) in enumerate(pairs):
            exp = orc.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md)
            got = out[:, starts[p]:starts[p] + counts[p]].T
            assert got.shape == exp.shape and (got == exp).all(), (ratio, cc, md, p)
            assert (got == matcher.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md, bits)).all(), (ratio, cc, md, p)
        assert counts[0] > 0
    # one query row more, or one train row more, and the pair no longer fits
    for offs_big in ([0, n1 + 1, n1 + 1 + n2], [0, n1, n1 + 1, n1 + 2 + n2]):
        offs_big = np.array(offs_big, dtype=np.int64)
        with pytest.raises(PgmatchError) as ei:
            matcher.match_ratio_crosscheck_batch_dev(d_all, offs_big, [(0, len(offs_big) - 2)], bits)
        assert ei.value.status == PGM_E_INVALID_ARG
    # one query row less still fits (and the handle works after the refused calls)
    offs_small = np.array([0, n1 - 1, n1 + 1, n1 + 1 + n2], dtype=np.int64)
    out, starts, counts = matcher.match_ratio_crosscheck_batch_dev(d_all, offs_small, [(0, 2)], bits, 0.9, False, -1)
    exp = orc.match_ratio_crosscheck(q[:n1 - 1], t[:n2], 0.9, False, -1)
    assert counts[0] > 0 and (out[:, :counts[0]].T.cpu().numpy() == exp).all()


# --- 7. train-sharded paths ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("shards", [3, 8])
@pytest.mark.parametrize("bits,stride", WIDE, ids=[_wid(w) for w in WIDE])
def test_train_sharded_emulated_per_width(matcher, bits, stride, shards):
    import torch
    q = _uniform(bits + 70, 3000, bits, stride)
    t = _noisy(bits + 71, _uniform(bits + 70, 3000, bits, stride), bits)[:2500]
    t[5:9] = t[5]
    exp = orc.match_sweep(q, t)
    outs, rounds = sharding.match_train_sharded_emulated(matcher, q, t, shards, desc_bits=bits)
    assert rounds > 0
    for o in outs:
        assert o.shape == exp.shape and (o == exp).all()
    dev = torch.device("cuda", matcher.device)
    d_q, d_t = torch.from_numpy(q).to(dev), torch.from_numpy(t).to(dev)
    for ratio, cc, md in RATIO_GRID[:3]:
        knn, kept = sharding.knn_train_sharded_emulated(matcher, d_q, d_t, shards, bits, ratio, cc, md)
        for a, b in zip(knn, orc.knn2(q, t)):
            assert (a.cpu().numpy() == b).all()
        got = kept.cpu().numpy().T
        exp_rc = orc.match_ratio_crosscheck(q, t, ratio, cc, md)
        assert got.shape == exp_rc.shape and (got == exp_rc).all(), (ratio, cc, md)


@pytest.mark.timeout(400)
@pytest.mark.parametrize("bits,stride", WIDE, ids=[_wid(w) for w in WIDE])
def test_multi_gpu_matcher_world_of_one_per_width(matcher, bits, stride):
    import torch
    # 30000 x 29000: the rounds, then the replicated finish; the small ones finish right after round 0
    for n1, n2, dist in [(5000, 4200, "U"), (3000, 3000, "C"), (1500, 40, "U"), (30000, 29000, "U")]:
        q, t = _pair(bits + 80 + n1, n1, n2, dist, bits, stride)
        exp = orc.match_rounds(q, t) if n1 * n2 > 10 ** 8 else orc.match_sweep(q, t)
        assert (matcher.match_greedy(q, t, bits) == exp).all()
        mg = sharding.MultiGpuMatcher(matcher, 0, 1)
        try:
            d_q, d_t = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
            got = mg.match_train_sharded(d_q, d_t, 0, n2, desc_bits=bits).T.cpu().numpy()
            assert got.shape == exp.shape and (got == exp).all(), (n1, n2)
            knn = mg.knn2_train_sharded(d_q, d_t, 0, desc_bits=bits)
            assert all((a.cpu().numpy() == b).all() for a, b in zip(knn, orc.knn2(q, t)))
        finally:
            mg.close()


# --- 8. the producer chain at NumGaussianPairs other than 256 -----------------------------------------------------

@pytest.mark.parametrize("n_pairs", [128, 384, 512])
def test_detect_describe_into_greedy_per_width(matcher, n_pairs):
    import torch
    g = np.load(os.path.join(GOLDEN, "lego_crop_detect.npz"))
    th = float(g["threshold"])
    pairs = D.gaussian_pairs(17, n_pairs, 50)
    stride = ((n_pairs + 127) // 128) * 16
    dev = torch.device("cuda", matcher.device)
    descs, exp_descs = [], []
    for k in (0, 1):
        gray = np.ascontiguousarray(g[f"gray{k}"], dtype=np.float32)
        xy, _, desc = matcher.detect_describe_dev(torch.from_numpy(gray).to(dev), th, pairs.reshape(-1, 4),
                                                  python_generation=True)
        exy, _ = D.detect_vectorised(gray, th, True)
        assert len(exy) > 2000 and xy.shape == exy.shape and (xy.cpu().numpy() == exy).all()
        exp = pack_descriptors(D.brief_descriptors(gray, exy, pairs, lsb_first=True), n_pairs)
        assert desc.shape == exp.shape == (len(exy), stride) and (desc.cpu().numpy() == exp).all()
        descs.append(desc.contiguous())
        exp_descs.append(exp)
    n1, n2 = len(exp_descs[0]), len(exp_descs[1])
    o = torch.empty((3, n1), dtype=torch.int32, device=dev)
    with matcher.torch_ordered():
        cnt = matcher.match_greedy_dev(descs[0].data_ptr(), n1, descs[1].data_ptr(), n2, n_pairs, stride,
                                       o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), n1)
    torch.cuda.synchronize()
    assert cnt == n1
    assert (o.T.cpu().numpy() == orc.match_sweep(exp_descs[0], exp_descs[1])).all()


# --- 9. argument checks -------------------------------------------------------------------------------------------

BAD_FORMATS = [(256, 0), (256, 8), (256, 80), (256, 128), (0, 32), (513, 64), (300, 32)]


def test_every_entry_point_rejects_bad_formats(matcher):
    # straight through the C ABI: the numpy wrappers would pad an 8-byte row and replace desc_bits = 0 by the row width.
    # Every buffer holds n = 4 rows of 128 bytes, so a check that let a format through would still read in bounds.
    import torch
    lib, h = matcher._lib, matcher._h
    n = 4
    host = np.zeros((2 * n, 128), dtype=np.uint8)
    hq, ht = host.ctypes.data, host[n:].ctypes.data
    hout = np.zeros((4, 2 * n * n), dtype=np.int64)
    o = [hout[k].ctypes.data for k in range(4)]
    dev = torch.zeros((2 * n, 128), dtype=torch.uint8, device="cuda")
    dq, dt = dev.data_ptr(), dev[n:].data_ptr()
    dout = torch.zeros((4, 2 * n * n), dtype=torch.int64, device="cuda")
    do = [dout[k].data_ptr() for k in range(4)]
    offs = np.array([0, n, 2 * n], dtype=np.int64)
    pl = np.array([[0, 1]], dtype=np.int32)
    counts = np.zeros(1, dtype=np.int32)
    cnt = C.c_int32(0)
    flag = PGM_FLAG_REFERENCE_COMPAT_TAIL
    calls = {
        "greedy": lambda b, s: lib.pgm_match_hamming_greedy(h, hq, n, ht, n, b, s, o[0], o[1], o[2], n, C.byref(cnt), flag),
        "greedy_dev": lambda b, s: lib.pgm_match_hamming_greedy_dev(h, dq, n, dt, n, b, s, do[0], do[1], do[2], n,
                                                                    C.byref(cnt), flag),
        "batch": lambda b, s: lib.pgm_match_pairs_batch(h, hq, offs.ctypes.data, 2, pl.ctypes.data, 1, b, s, o[0], o[1],
                                                        o[2], n, counts.ctypes.data, flag),
        "batch_dev": lambda b, s: lib.pgm_match_pairs_batch_dev(h, dq, offs.ctypes.data, 2, pl.ctypes.data, 1, b, s, do[0],
                                                                do[1], do[2], n, counts.ctypes.data, flag),
        "knn2": lambda b, s: lib.pgm_knn2_hamming(h, hq, n, ht, n, b, s, o[0], o[1], o[2], o[3]),
        "knn2_dev": lambda b, s: lib.pgm_knn2_hamming_dev(h, dq, n, dt, n, b, s, do[0], do[1], do[2], do[3]),
        "ratio": lambda b, s: lib.pgm_match_ratio_crosscheck(h, hq, n, ht, n, b, s, 0.8, 1, -1, o[0], o[1], o[2], n,
                                                             C.byref(cnt)),
        "sorted": lambda b, s: lib.pgm_match_keypoints_sorted(h, hq, n, ht, n, b, s, o[0]),
        "sorted_dev": lambda b, s: lib.pgm_match_keypoints_sorted_dev(h, dq, n, dt, n, b, s, do[0]),
        "ratio_batch": lambda b, s: lib.pgm_match_ratio_crosscheck_batch_dev(h, dq, offs.ctypes.data, 2, pl.ctypes.data, 1,
                                                                             b, s, 0.8, 1, -1, do[0], do[1], do[2], 2 * n,
                                                                             counts.ctypes.data),
    }

    def shard(b, s):
        sh = C.c_void_p()
        rc = lib.pgm_shard_create(h, dq, n, dt, n, 0, n, b, s, C.byref(sh))
        if sh.value:
            lib.pgm_shard_destroy(sh)
        return rc
    calls["shard"] = shard
    bad = [(name, b, s, rc) for name, f in calls.items() for b, s in BAD_FORMATS if (rc := f(b, s)) != PGM_E_INVALID_ARG]
    assert not bad, bad
    torch.cuda.synchronize()
    # the handle is still usable, and the same buffers with a valid format go through every family
    for name, f in calls.items():
        assert f(256, 32) == 0, name
    q, t = _pair(3, 300, 200, "U", 512, 64)
    assert (matcher.match_greedy(q, t, 512) == orc.match_sweep(q, t)).all()
