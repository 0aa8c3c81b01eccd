"""Ratio test + cross-check for many pairs of any size (pgm_match_ratio_crosscheck_pairs_batch_dev; run on a B200: -m gpu).

Every comparison is bit-exact.  Expected values come from the oracle (orc.match_ratio_crosscheck), from the per-pair entry
point pgm_match_ratio_crosscheck and, for pairs within its shared-memory bound, from the one-CTA-per-pair batch
(pgm_match_ratio_crosscheck_batch_dev)."""
import numpy as np
import pytest

from oracle import orc
from photogrammetry_b200 import sharding, synthetic
from photogrammetry_b200._lib import PGM_E_CAPACITY, PGM_E_INVALID_ARG, PgmatchError

pytestmark = pytest.mark.gpu

# the row widths of test_gpu_widths.py: every instantiation, a partial last word, 256 bits in rows wider than needed
WIDTHS = [(64, 16), (128, 16), (200, 32), (300, 48), (384, 48), (512, 64), (256, 64)]
RATIO_GRID = [(0.8, True, -1), (0.9, False, -1), (0.0, True, -1), (0.0, False, 75), (0.7, True, 60)]
RCB_SMEM_MAX = 200 * 1024
ORACLE_MAX_CELLS = 20_000_000      # larger pairs: the oracle at the first grid point, the per-pair call at every point


@pytest.fixture(scope="module")
def torch_dev(matcher):
    import torch
    return torch.device("cuda", matcher.device)


def _wid(w):
    return f"{w[0]}b{w[1]}B"


def _images(sizes, bits, stride, seed):
    """Images that share content: image k is a noisy copy of the first rows of one base set, so matches survive."""
    base = synthetic.uniform_descriptors(seed, max(sizes), bits, stride)
    imgs = [base[:n] if k % 2 == 0 else synthetic.noisy_copy_descriptors(seed + 1 + k, base, bits)[:n]
            for k, n in enumerate(sizes)]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return imgs, np.concatenate(imgs), offs


def _per_pair(out, starts, counts, p):
    out = out if isinstance(out, np.ndarray) else out.cpu().numpy()
    return out[:, starts[p]:starts[p] + counts[p]].T


def _fits_one_cta(n1, n2, stride):
    return (n1 + n2) * stride + 4 * n2 + 16 <= RCB_SMEM_MAX


# --- 1. every width, images of 0 .. 20 000 rows ----------------------------------------------------------------------

SIZES = [0, 1, 500, 600, 3000, 5000, 20000]
# both directions, a self pair, a repeated pair, n2 = 1, n2 = 0 and n1 = 0
PAIRS = [(2, 3), (3, 2), (4, 5), (5, 4), (6, 4), (4, 6), (3, 3), (2, 3), (5, 1), (1, 5), (1, 1), (4, 0), (0, 4), (2, 4)]


@pytest.mark.timeout(900)
@pytest.mark.parametrize("bits,stride", WIDTHS, ids=[_wid(w) for w in WIDTHS])
def test_pairs_batch_every_width(matcher, torch_dev, bits, stride):
    import torch
    imgs, all_desc, offs = _images(SIZES, bits, stride, bits * 11 + stride)
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    pairs = np.array(PAIRS, dtype=np.int32)
    small = [p for p, (a, b) in enumerate(PAIRS) if _fits_one_cta(SIZES[a], SIZES[b], stride)]
    for g, (ratio, cc, md) in enumerate(RATIO_GRID):
        out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, bits, ratio, cc, md)
        out = out.cpu().numpy()
        assert (starts == np.concatenate([[0], np.cumsum([SIZES[a] for a, _ in PAIRS])[:-1]])).all()
        for p, (a, b) in enumerate(PAIRS):
            got = _per_pair(out, starts, counts, p)
            one = matcher.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md, bits)
            assert got.shape == one.shape and (got == one).all(), (ratio, cc, md, p)
            if SIZES[a] * SIZES[b] <= ORACLE_MAX_CELLS or g == 0:
                exp = orc.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md)
                assert got.shape == exp.shape and (got == exp).all(), (ratio, cc, md, p)
            if SIZES[a] == 0 or SIZES[b] == 0:
                assert counts[p] == 0
        assert counts[PAIRS.index((4, 5))] > 0 and (counts[0] == counts[7]) and (_per_pair(out, starts, counts, 0) == _per_pair(out, starts, counts, 7)).all()
        # pairs within the one-CTA kernel's bound: the same output, counts included
        so, ss, sc = matcher.match_ratio_crosscheck_batch_dev(d_all, offs, pairs[small], bits, ratio, cc, md)
        for k, p in enumerate(small):
            assert sc[k] == counts[p], (ratio, cc, md, p)
            assert (_per_pair(so, ss, sc, k) == _per_pair(out, starts, counts, p)).all(), (ratio, cc, md, p)


# --- 2. heavy ties: 8-bit descriptors ----------------------------------------------------------------------------------

def test_heavy_ties_8_bit(matcher, torch_dev):
    """256 possible descriptors over 3 000 x 3 000 rows: every distance, best and column minimum is tied many times over,
    and the duplicates of each train row fall into different column splits and row tiles of the fused pass."""
    import torch
    bits, stride, n = 8, 16, 3000
    q = synthetic.uniform_descriptors(801, n, bits, stride)
    t = synthetic.uniform_descriptors(802, n, bits, stride)
    t[2900:] = t[:100]                               # exact duplicates 2 900 columns apart (other splits)
    q[2500:2600] = q[:100]                           # duplicated queries in other row tiles
    d_all = torch.from_numpy(np.concatenate([q, t])).to(torch_dev)
    offs = np.array([0, n, 2 * n], dtype=np.int64)
    pairs = np.array([(0, 1), (1, 0), (0, 0)], dtype=np.int32)
    imgs = [q, t]
    for ratio, cc, md in RATIO_GRID + [(0.0, True, 0)]:
        out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, bits, ratio, cc, md)
        for p, (a, b) in enumerate(pairs):
            got = _per_pair(out, starts, counts, p)
            exp = orc.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md)
            assert got.shape == exp.shape and (got == exp).all(), (ratio, cc, md, p)
            assert (got == matcher.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md, bits)).all()
        if cc and ratio == 0.0:
            assert counts.min() > 0


# --- 3. one large pair ---------------------------------------------------------------------------------------------------

@pytest.mark.timeout(600)
def test_one_large_pair(matcher, torch_dev):
    """60 000 x 50 000 at 256 bits: 118 row tiles, so the columns are split (about two waves of CTAs)."""
    import torch
    bits, stride, n1, n2 = 256, 32, 60000, 50000
    q = synthetic.uniform_descriptors(901, n1, bits, stride)
    t = synthetic.noisy_copy_descriptors(902, q, bits)[:n2].copy()
    t[40000:40010] = t[10]                           # duplicates far apart: different column splits
    d_all = torch.from_numpy(np.concatenate([q, t])).to(torch_dev)
    offs = np.array([0, n1, n1 + n2], dtype=np.int64)
    for ratio, cc, md in [(0.8, True, -1), (0.0, False, 80), (0.7, True, 60)]:
        out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, [(0, 1)], bits, ratio, cc, md)
        st = matcher.stats()
        exp = matcher.match_ratio_crosscheck(q, t, ratio, cc, md, bits)
        got = _per_pair(out, starts, counts, 0)
        assert counts[0] > 1000 and got.shape == exp.shape and (got == exp).all(), (ratio, cc, md)
        assert st["distance_evals"] == st["evals_computed"] == n1 * n2 and st["kernel_launches"] == 3


# --- 4. chunking ---------------------------------------------------------------------------------------------------------

def test_chunks_of_many_small_pairs(matcher, torch_dev):
    """5 000 pairs are more than one chunk (<= 4 096 pairs each): three launches per chunk, same output as the one-CTA
    batch, and each chunk writes at its own offsets."""
    import torch
    bits, stride, per, n_img = 256, 32, 64, 100
    imgs, all_desc, offs = _images([per] * n_img, bits, stride, 1001)
    pairs = sharding.all_pairs(n_img)                       # 4 950 pairs, then 50 of them again
    pairs = np.concatenate([pairs, pairs[:50]]).astype(np.int32)
    assert len(pairs) == 5000
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    for ratio, cc, md in RATIO_GRID[:2]:
        out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, bits, ratio, cc, md)
        st = matcher.stats()
        assert st["kernel_launches"] == 6 and st["pairs"] == 5000 and st["matched"] == counts.sum()
        so, ss, sc = matcher.match_ratio_crosscheck_batch_dev(d_all, offs, pairs, bits, ratio, cc, md)
        assert (ss == starts).all() and (sc == counts).all() and counts.sum() > 0
        out, so = out.cpu().numpy(), so.cpu().numpy()
        for p in range(len(pairs)):
            assert (_per_pair(out, starts, counts, p) == _per_pair(so, ss, sc, p)).all(), p


@pytest.mark.timeout(600)
def test_64_images_of_4096(matcher, torch_dev):
    import torch
    bits, stride, per, n_img = 256, 32, 4096, 64
    imgs, all_desc, offs = _images([per] * n_img, bits, stride, 1101)
    pairs = sharding.all_pairs(n_img)
    assert len(pairs) == 2016
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, bits, 0.8, True, -1)
    st = matcher.stats()
    assert st["distance_evals"] == st["evals_computed"] == 2016 * per * per and st["host_syncs"] <= 2
    out = out.cpu().numpy()
    for p in np.linspace(0, len(pairs) - 1, 64).astype(int):
        a, b = pairs[p]
        exp = matcher.match_ratio_crosscheck(imgs[a], imgs[b], 0.8, True, -1, bits)
        got = _per_pair(out, starts, counts, p)
        assert got.shape == exp.shape and (got == exp).all(), p
    assert counts.sum() > 0


# --- 5. statistics -------------------------------------------------------------------------------------------------------

def test_statistics(matcher, torch_dev):
    import torch
    bits, stride = 256, 32
    sizes = [700, 0, 1300, 2100]
    imgs, all_desc, offs = _images(sizes, bits, stride, 1201)
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    pairs = [(0, 2), (2, 3), (1, 3), (3, 1), (3, 0)]
    evals = sum(sizes[a] * sizes[b] for a, b in pairs)
    for cc in (True, False):
        out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, bits, 0.8, cc, -1)
        st = matcher.stats()
        assert st["distance_evals"] == st["evals_computed"] == evals
        assert st["host_syncs"] <= 2 and st["pairs"] == len(pairs) and st["matched"] == counts.sum() > 0
        assert st["kernel_launches"] == 3


# --- 6. output contract --------------------------------------------------------------------------------------------------

def test_slots_after_count_keep_their_sentinel(matcher, torch_dev):
    import torch
    bits, stride = 256, 32
    sizes = [900, 1100, 5000]
    imgs, all_desc, offs = _images(sizes, bits, stride, 1301)
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    pairs = np.array([(0, 1), (1, 2), (2, 0), (2, 1)], dtype=np.int32)
    total = sum(sizes[a] for a, _ in pairs)
    sentinel = -12345
    out = torch.full((3, total), sentinel, dtype=torch.int32, device=torch_dev)
    counts = np.zeros(len(pairs), dtype=np.int32)
    lib = matcher._lib
    with matcher.torch_ordered():
        rc = lib.pgm_match_ratio_crosscheck_pairs_batch_dev(matcher._h, d_all.data_ptr(), offs.ctypes.data, len(sizes),
                                                            pairs.ctypes.data, len(pairs), bits, stride, 0.8, 1, -1,
                                                            out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                                            total, counts.ctypes.data)
    assert rc == 0
    o = out.cpu().numpy()
    start = 0
    for p, (a, b) in enumerate(pairs):
        exp = orc.match_ratio_crosscheck(imgs[a], imgs[b], 0.8, True, -1)
        assert counts[p] == len(exp) and 0 < counts[p] < sizes[a]
        assert (o[:, start:start + counts[p]].T == exp).all()
        assert (o[:, start + counts[p]:start + sizes[a]] == sentinel).all(), p
        start += sizes[a]


# --- 7. errors -----------------------------------------------------------------------------------------------------------

def test_errors_leave_the_handle_usable(matcher, torch_dev):
    import torch
    bits, stride = 256, 32
    sizes = [300, 400]
    imgs, all_desc, offs = _images(sizes, bits, stride, 1401)
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    out = torch.empty((3, 1000), dtype=torch.int32, device=torch_dev)
    counts = np.zeros(4, dtype=np.int32)
    lib, h = matcher._lib, matcher._h

    def call(offs_, pairs_, cap=1000, b=bits, s=stride):
        offs_ = np.ascontiguousarray(offs_, dtype=np.int64)
        pairs_ = np.ascontiguousarray(pairs_, dtype=np.int32)
        return lib.pgm_match_ratio_crosscheck_pairs_batch_dev(h, d_all.data_ptr(), offs_.ctypes.data, len(offs_) - 1,
                                                              pairs_.ctypes.data, len(pairs_), b, s, 0.8, 1, -1,
                                                              out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                                              cap, counts.ctypes.data)
    assert call(offs, [(0, 1), (1, 0)], cap=699) == PGM_E_CAPACITY
    assert call(offs, [(0, 2)]) == PGM_E_INVALID_ARG                       # pair index out of range
    assert call(offs, [(0, 1), (-1, 0)]) == PGM_E_INVALID_ARG
    assert call([0, 300, 200], [(0, 1)]) == PGM_E_INVALID_ARG             # decreasing offsets
    assert call([0, 1 << 20, (1 << 20) + 10], [(1, 0)]) == PGM_E_INVALID_ARG   # a size >= 2^20
    for b, s in [(256, 8), (0, 32), (300, 32), (513, 64)]:
        assert call(offs, [(0, 1)], b=b, s=s) == PGM_E_INVALID_ARG
    with pytest.raises(PgmatchError) as ei:
        matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, [(0, 5)], bits)
    assert ei.value.status == PGM_E_INVALID_ARG
    torch.cuda.synchronize()
    got, starts, cnt = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, [(0, 1), (1, 0)], bits, 0.8, True, -1)
    for p, (a, b) in enumerate([(0, 1), (1, 0)]):
        assert (_per_pair(got, starts, cnt, p) == orc.match_ratio_crosscheck(imgs[a], imgs[b], 0.8, True, -1)).all()
    assert cnt.sum() > 0


# --- 8. pair sharding ----------------------------------------------------------------------------------------------------

def test_pair_sharded_blocks_equal_one_call(matcher, torch_dev):
    import torch
    bits, stride = 256, 32
    sizes = [900, 2500, 0, 1800, 4100, 300, 3000, 1200]
    imgs, all_desc, offs = _images(sizes, bits, stride, 1501)
    d_all = torch.from_numpy(all_desc).to(torch_dev)
    pairs = sharding.all_pairs(len(sizes))
    out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, bits, 0.8, True, -1)
    ref = [_per_pair(out, starts, counts, p) for p in range(len(pairs))]
    for world in (2, 3, 8):
        got_counts, got = [], []
        for rank in range(world):
            lo, hi = sharding.shard_for_rank(pairs, np.diff(offs), rank, world)
            o, s, c = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs[lo:hi], bits, 0.8, True, -1)
            got_counts.append(c)
            got += [_per_pair(o, s, c, p) for p in range(hi - lo)]
        assert (np.concatenate(got_counts) == counts).all(), world
        assert len(got) == len(ref) and all((x == y).all() for x, y in zip(got, ref)), world


# --- 9. streams ----------------------------------------------------------------------------------------------------------

def test_on_a_non_default_torch_stream(matcher, torch_dev):
    """Inputs written by a torch kernel on a side stream and outputs consumed there, with no synchronisation between."""
    import torch
    bits, stride = 256, 32
    sizes = [4000, 3500]
    imgs, all_desc, offs = _images(sizes, bits, stride, 1601)
    host = torch.from_numpy(all_desc).pin_memory()
    mask = torch.full((1, stride), 0xFF, dtype=torch.uint8, device=torch_dev)
    side = torch.cuda.Stream(device=torch_dev)
    with torch.cuda.stream(side):
        d_all = host.to(torch_dev, non_blocking=True)
        d_all = (d_all ^ mask) ^ mask                         # written by torch kernels on the side stream
        out, starts, counts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, [(0, 1), (1, 0)], bits)
        n = int(counts[0])
        tj = out[1, :n].to(torch.int64)
        d = d_all[int(offs[1]):][tj] ^ d_all[:int(offs[1])][out[0, :n].to(torch.int64)]   # consumed on the side stream
        ok = (out[2, :n] > -1).all()
    side.synchronize()
    assert bool(ok)
    exp = orc.match_ratio_crosscheck(imgs[0], imgs[1], 0.8, True, -1)
    assert n == len(exp) > 0 and (out[:, :n].T.cpu().numpy() == exp).all()
    assert (np.bitwise_count(d.cpu().numpy()).sum(axis=1) == exp[:, 2]).all()
