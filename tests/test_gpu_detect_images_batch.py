"""pgm_detect_describe_images_batch_dev: FAST-12 -> (NMS) -> BRIEF for a set of device-resident images of different
sizes in one call.  Per image the result must equal pgm_detect_describe_dev on that image alone, bit for bit
(coordinates, FastScore, descriptor bytes, order, count); a set of equal images must equal the uniform batch forms;
and image_set.match_image_set_dev must equal the oracle chain from pixels to RANSAC."""
import numpy as np
import pytest

from oracle import detect_np as D
from oracle import orc
from oracle import ransac_batch_np as R
from photogrammetry_b200 import image_set, sequence, synthetic
from photogrammetry_b200._lib import PGM_E_INVALID_ARG, PGM_FLAG_PYTHON_GENERATION, PGM_OK
from photogrammetry_b200.descriptors import pack_descriptors
from photogrammetry_b200.sharding import all_pairs

pytestmark = pytest.mark.gpu

CS_PAIRS = D.gaussian_pairs(11, 256, 50)
CS_TABLE = CS_PAIRS.reshape(-1, 4).astype(np.int32)
PY_TABLE = sequence.pairs_table(sequence.star_pairs())
SENTINEL = -7


def _mixed_set(pg):
    """Landscape and portrait 4000 x 3000, odd widths, images without a FAST interior (7 x 7, 6 x 200, 200 x 6, 1 x 1),
    the dotted-row chain frame (hundreds of NMS rounds at r = 4) and two star frames, on the generation's scale."""
    scale = 255.0 if pg else 1.0
    rng = np.random.default_rng(5)
    star = sequence.shifted_frames(sequence.star_gray(), 2, 40).astype(np.float32)
    ims = [synthetic.rectangles_image(3000, 4000, seed=7), synthetic.rectangles_image(4000, 3000, seed=8),
           synthetic.rectangles_image(217, 333, seed=9), rng.random((7, 7), dtype=np.float32),
           rng.random((95, 1001), dtype=np.float32), rng.random((200, 6), dtype=np.float32),
           rng.random((6, 200), dtype=np.float32), np.ones((1, 1), np.float32),
           synthetic.dotted_row_image(), synthetic.rectangles_image(129, 65, seed=10)]
    ims = [np.ascontiguousarray(im * np.float32(scale)) for im in ims]
    star = star if pg else star / np.float32(255.0)
    return ims + [star[0], star[1]], (50.0 if pg else 0.1)


def _pack(images, gap=0, fill=np.nan):
    """One flat device buffer with `gap` pixels of `fill` before, between and after the images (fill None: a
    checkerboard of 0 and 1e4, which makes corners wherever it is read)."""
    import torch
    sizes = [im.size for im in images]
    offs = np.zeros(len(images) + 1, np.int64)
    for k, s in enumerate(sizes):
        offs[k + 1] = offs[k] + s + gap
    offs += gap
    total = int(offs[-1]) + gap
    if fill is None:
        buf = np.where(np.arange(total) % 2 == 0, 0.0, 1e4).astype(np.float32)
    else:
        buf = np.full(total, fill, np.float32)
    for k, im in enumerate(images):
        buf[offs[k]:offs[k] + im.size] = im.reshape(-1)
    return torch.from_numpy(buf).cuda(), offs


def _call(matcher, d_buf, offs, images, th, r, cap, pg=False, table=CS_TABLE, read_counts=True, stride=32, **over):
    """The C ABI into outputs pre-filled with a sentinel, one image's slots more than needed."""
    import torch
    k = len(images)
    dev = d_buf.device
    w = np.array([im.shape[1] for im in images], np.int32)
    h = np.array([im.shape[0] for im in images], np.int32)
    offs = np.ascontiguousarray(offs, np.int64)
    out = (torch.full((k + 1, cap, 2), SENTINEL, dtype=torch.int32, device=dev),
           torch.full((k + 1, cap), SENTINEL, dtype=torch.int32, device=dev),
           torch.full((k + 1, cap, stride), 0xA5, dtype=torch.uint8, device=dev),
           torch.full((k + 1,), SENTINEL, dtype=torch.int32, device=dev))
    h_cnt = np.full(k + 1, SENTINEL, dtype=np.int32)
    a = dict(gray=d_buf.data_ptr(), pix_offs=offs.ctypes.data, w=w.ctypes.data, h=h.ctypes.data, n=k,
             pairs=table.ctypes.data, n_pairs=len(table), capacity=cap, xy=out[0].data_ptr(), sc=out[1].data_ptr(),
             desc=out[2].data_ptr(), cnt=out[3].data_ptr())
    a.update(over)
    with matcher.torch_ordered(dev):
        rc = matcher._lib.pgm_detect_describe_images_batch_dev(
            matcher._h, a["gray"], a["pix_offs"], a["w"], a["h"], a["n"], float(th), int(r), a["pairs"], a["n_pairs"],
            stride, PGM_FLAG_PYTHON_GENERATION if pg else 0, a["xy"], a["sc"], a["desc"], a["capacity"], a["cnt"],
            h_cnt.ctypes.data if read_counts else None)
    return rc, tuple(x.cpu().numpy() for x in out), h_cnt


def _per_image(matcher, images, th, table, r, pg):
    import torch
    return [tuple(x.cpu().numpy() for x in matcher.detect_describe_dev(torch.from_numpy(im).cuda(), th, table, nms_radius=r,
                                                                      python_generation=pg, capacity=65536))
            for im in images]


def _assert_equal(out, exp, cap):
    xy, sc, desc, counts = out
    for k, (exy, esc, edesc) in enumerate(exp):
        n = len(exy)
        m = min(n, cap)
        assert int(counts[k]) == n, (k, int(counts[k]), n)
        assert (xy[k, :m] == exy[:m]).all() and (sc[k, :m] == esc[:m]).all() and (desc[k, :m] == edesc[:m]).all(), k
        assert (xy[k, m:] == SENTINEL).all() and (sc[k, m:] == SENTINEL).all() and (desc[k, m:] == 0xA5).all(), k
    assert (xy[len(exp)] == SENTINEL).all() and (desc[len(exp)] == 0xA5).all() and counts[len(exp)] == SENTINEL


@pytest.mark.parametrize("r", [-1, 0, 1, 4, 10])
@pytest.mark.parametrize("pg", [False, True])
def test_mixed_set_equals_per_image_calls(matcher, pg, r):
    images, th = _mixed_set(pg)
    table = PY_TABLE if pg else CS_TABLE
    exp = _per_image(matcher, images, th, table, r, pg)
    assert all(len(exp[k][0]) == 0 for k in (5, 6, 7))                # no FAST interior
    assert len(exp[0][0]) > 1000 and len(exp[1][0]) > 1000 and len(exp[8][0]) > 0
    for gap, fill in ((0, 0.0), (37, np.nan), (53, None)):             # only the declared pixels are read
        d_buf, offs = _pack(images, gap, fill)
        rc, out, h_cnt = _call(matcher, d_buf, offs, images, th, r, 65536, pg=pg, table=table)
        assert rc == PGM_OK
        assert (h_cnt[:len(images)] == out[3][:len(images)]).all()
        _assert_equal(out, exp, 65536)
    st = matcher.stats()
    assert (st["host_syncs"], st["kernel_launches"]) == ((1, 6) if r < 0 else (2, 11))


def test_chain_frame_rounds_next_to_large_images(matcher):
    """The dotted row needs 496 rounds at r = 4; next to 4000 x 3000 images it must still give 248 survivors."""
    images, th = _mixed_set(False)
    d_buf, offs = _pack(images)
    rc, out, _ = _call(matcher, d_buf, offs, images, th, 4, 8192)
    assert rc == PGM_OK and out[3][8] == 248
    exy, esc = D.detect_vectorised(images[8], th)
    kept = D.eliminate_redundant_vectorised(exy, esc, 4)
    assert (out[0][8, :248] == exy[kept]).all()
    assert (out[2][8, :248] == pack_descriptors(D.brief_descriptors(images[8], exy[kept], CS_PAIRS), 256)).all()


@pytest.mark.parametrize("r", [-1, 10])
def test_equal_sizes_equal_uniform_forms(matcher, r):
    import torch
    frames = sequence.shifted_frames(sequence.star_gray(), 32, 5).astype(np.float32)
    d = torch.from_numpy(frames).cuda()
    ref = [x.cpu().numpy() if hasattr(x, "cpu") else x
           for x in matcher.detect_describe_batch_dev(d, 50.0, PY_TABLE, capacity=256, python_generation=True, nms_radius=r)]
    ref_st = matcher.stats()
    got = [x.cpu().numpy() if hasattr(x, "cpu") else x
           for x in matcher.detect_describe_images_batch_dev(list(d), 50.0, PY_TABLE, capacity=256,
                                                             python_generation=True, nms_radius=r)]
    st = matcher.stats()
    assert (got[3] == ref[3]).all() and (ref[3] > 0).all()
    for k, n in enumerate(ref[3]):
        for g, e in zip(got[:3], ref[:3]):
            assert (g[k, :n] == e[k, :n]).all(), k
    assert (st["host_syncs"], st["kernel_launches"]) == (ref_st["host_syncs"], ref_st["kernel_launches"])


@pytest.mark.parametrize("r", [-1, 4])
def test_capacity_truncation(matcher, r):
    """Images with more survivors than capacity: the first `capacity` slots are right, the count is the full one, and
    nothing at or beyond min(count, capacity) is written."""
    images, th = _mixed_set(False)
    images = images[2:]                                                  # without the 4000 x 3000 pair
    exp = _per_image(matcher, images, th, CS_TABLE, r, False)
    counts = [len(e[0]) for e in exp]
    cap = 127
    assert max(counts) > cap and 0 < min(c for c in counts if c) < cap
    for read_counts in (True, False):
        d_buf, offs = _pack(images, 11, None)
        rc, out, h_cnt = _call(matcher, d_buf, offs, images, th, r, cap, read_counts=read_counts)
        assert rc == PGM_OK
        _assert_equal(out, exp, cap)
        if read_counts:
            assert (h_cnt[:len(images)] == counts).all()
        st = matcher.stats()
        assert st["host_syncs"] == (r >= 0) + read_counts


@pytest.mark.parametrize("n_images", [1, 3, 64])
def test_syncs_and_launches_independent_of_set(matcher, n_images):
    rng = np.random.default_rng(n_images)
    images = [rng.random((int(rng.integers(8, 300)), int(rng.integers(8, 300))), dtype=np.float32)
              for _ in range(n_images)]
    d_buf, offs = _pack(images, 3)
    for r, read_counts, want in ((-1, False, (0, 6)), (-1, True, (1, 6)), (3, False, (1, 11)), (3, True, (2, 11))):
        rc, out, _ = _call(matcher, d_buf, offs, images, 0.1, r, 2048, read_counts=read_counts)
        assert rc == PGM_OK and (out[3][:n_images] > 0).all()
        st = matcher.stats()
        assert (st["host_syncs"], st["kernel_launches"]) == want, (r, read_counts)


def test_refusals_then_a_correct_call(matcher):
    images, th = _mixed_set(False)
    images = images[2:5]
    d_buf, offs = _pack(images, 5)
    exp = _per_image(matcher, images, th, CS_TABLE, 2, False)
    bad_w = np.array([333, 0, 1001], np.int32)
    big_w = np.array([333, 70000, 1001], np.int32)
    bad_h = np.array([217, 7, 0], np.int32)
    neg_offs = offs - 10
    tight = offs.copy()
    tight[2] = tight[1] + images[1].size - 1                               # image 1 overlaps image 2
    cases = [dict(gray=None), dict(pix_offs=None), dict(w=None), dict(h=None), dict(pairs=None), dict(xy=None),
             dict(sc=None), dict(desc=None), dict(cnt=None), dict(n=-1), dict(n=65536), dict(w=bad_w.ctypes.data),
             dict(w=big_w.ctypes.data), dict(h=bad_h.ctypes.data), dict(pix_offs=neg_offs.ctypes.data),
             dict(pix_offs=tight.ctypes.data), dict(capacity=0), dict(stride=24), dict(stride=16), dict(n_pairs=0)]
    for over in cases:
        stride = over.pop("stride", 32)
        rc, _, _ = _call(matcher, d_buf, offs, images, th, 2, 2048, stride=stride, **over)
        assert rc == PGM_E_INVALID_ARG, (over, stride)
        rc, out, _ = _call(matcher, d_buf, offs, images, th, 2, 2048)
        assert rc == PGM_OK, over
        _assert_equal(out, exp, 2048)
    rc, out, h_cnt = _call(matcher, d_buf, offs, images, th, 2, 2048, n=0)
    assert rc == PGM_OK and (h_cnt == SENTINEL).all() and (out[3] == SENTINEL).all() and (out[0] == SENTINEL).all()
    st = matcher.stats()
    assert st["host_syncs"] == 0 and st["kernel_launches"] == 0
    assert matcher._lib.pgm_detect_describe_images_batch_dev(None, None, None, None, None, 0, 0.1, 0, None, 0, 32, 0, None,
                                                             None, None, 1, None, None) == PGM_E_INVALID_ARG


def test_non_default_stream(matcher):
    import torch
    images, th = _mixed_set(True)
    images = images[2:]
    ref = matcher.detect_describe_images_batch_dev([torch.from_numpy(im).cuda() for im in images], th, PY_TABLE,
                                                   python_generation=True, nms_radius=10)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d = [torch.from_numpy(im).cuda() for im in images]
        got = matcher.detect_describe_images_batch_dev(d, th, PY_TABLE, python_generation=True, nms_radius=10,
                                                       read_counts=False)
        got = [x.cpu().numpy() for x in got]
    assert (got[3] == ref[3]).all() and ref[3].sum() > 0
    for k, n in enumerate(ref[3]):
        for g, r in zip(got[:3], ref[:3]):
            assert (g[k, :n] == r[k, :n].cpu().numpy()).all(), k


# ---- the image-set chain against the oracle chain ------------------------------------------------------------------
BOXES = [(0, 0, 640, 480), (180, 90, 480, 640), (300, 260, 800, 600), (90, 240, 600, 800), (520, 0, 701, 503),
         (40, 420, 517, 389)]
GAP_MIN, F_TOL, SIGN_MIN = 1e-8, 1e-6, 1e-9                 # tests/test_gpu_ransac_pairs.py states their reasons


@pytest.fixture(scope="module")
def crops_oracle():
    crops, origin = synthetic.scene_crops(21, BOXES)
    xy, desc = [], []
    for im in crops:
        f_xy, f_sc = D.detect_vectorised(im, 0.1)
        kept = D.eliminate_redundant_vectorised(f_xy, f_sc, 10)
        xy.append(f_xy[kept])
        desc.append(pack_descriptors(D.brief_descriptors(im, f_xy[kept], CS_PAIRS), 256))
    return crops, origin, xy, desc


@pytest.mark.parametrize("method", ["greedy", "ratio"])
def test_image_set_chain_equals_oracle(matcher, crops_oracle, method):
    import torch
    crops, origin, exy, edesc = crops_oracle
    plist = all_pairs(len(crops))
    S, P, thr = 2000, 32, 0.001
    res = image_set.match_image_set_dev(matcher, [torch.from_numpy(c).cuda() for c in crops], 0.1, CS_TABLE,
                                        nms_radius=10, method=method)
    assert len(res.pair_list) == 15
    xy_all, desc_all = res.xy.cpu().numpy(), res.desc.cpu().numpy()
    for k in range(len(crops)):
        o0, o1 = res.offsets[k], res.offsets[k + 1]
        assert int(res.counts[k]) == len(exy[k]) > 100
        assert (xy_all[o0:o1] == exy[k]).all() and (desc_all[o0:o1] == edesc[k]).all(), k
    matches = res.matches.cpu().numpy()
    for p, (a, b) in enumerate(plist):
        exp = orc.match_sweep(edesc[a], edesc[b]) if method == "greedy" else orc.match_ratio_crosscheck(edesc[a], edesc[b], 0.8, True)
        got = matches[:, res.starts[p]:res.starts[p] + res.match_counts[p]].T
        assert got.shape == exp.shape and (got == exp).all(), p

    # RANSAC: the chain's winner, inliers, F and mask, scored bit-exactly by the oracle on the device's own hypotheses,
    # and the device's F against the oracle's fp64 estimate of the same samples (up to sign where the sign is a tie)
    qi, tj = res.matches[0].contiguous(), res.matches[1].contiguous()
    hyp = matcher.ransac_fundamental_pairs_batch_dev(res.xy, res.offsets, plist, qi, tj, res.starts, res.match_counts,
                                                     n_samples=S, pairs_per_sample=P, threshold=thr, seed=0,
                                                     hypotheses=True)
    best, inl, F, mask, hF, hc = (x.cpu().numpy() for x in hyp)
    for got, ref in zip((res.best, res.inliers, res.F, res.mask), (best, inl, F, mask)):
        assert (got.cpu().numpy() == ref).all()
    qi, tj = qi.cpu().numpy(), tj.cpu().numpy()
    dev_true = dev_all = 0
    oracle = R.get_fundamental_pairs(xy_all, res.offsets, plist, qi, tj, res.starts, res.match_counts, S, P, thr, 0)
    or_true = or_all = 0
    for p, (a, b) in enumerate(plist):
        s, c = int(res.starts[p]), int(res.match_counts[p])
        if c < P:
            assert best[p] == -2 and oracle[p][0] == -2
            continue
        xy1 = xy_all[res.offsets[a] + qi[s:s + c].astype(np.int64)]
        xy2 = xy_all[res.offsets[b] + tj[s:s + c].astype(np.int64)]
        ec, eb, em = R.score(hF[p], R.rank2(hF[p]), xy1, xy2, thr)
        assert (hc[p] == ec).all() and best[p] == eb and inl[p] == em.sum() and (mask[s:s + c] == em).all(), p
        Fo = oracle[p][4]
        idx = np.stack([R.sample_indices(c, P, 0, int(a), int(b), k) for k in range(S)])
        _, sv = R.estimate(xy1[idx], xy2[idx], return_sv=True)
        keep = (sv[:, 7] - sv[:, 8]) / sv[:, 0] > GAP_MIN
        scale = np.abs(Fo).reshape(S, 9).max(1)
        err = np.abs(hF[p].astype(np.float64) - Fo).reshape(S, 9).max(1) / scale
        err_flip = np.abs(hF[p].astype(np.float64) + Fo).reshape(S, 9).max(1) / scale
        err = np.where(R.sign_margin(xy1[idx], xy2[idx]) < SIGN_MIN, np.minimum(err, err_flip), err)
        assert (err[keep] <= F_TOL).all(), (p, err[keep].max())
        # overlapping crops are a pure translation apart: count the winner's inliers that are true correspondences
        true = (xy2 == xy1 + (origin[a] - origin[b])).all(axis=1)
        if true.sum() >= P:
            dev_true += int((em.astype(bool) & true).sum()); dev_all += int(em.sum())
            om = oracle[p][3].astype(bool)
            or_true += int((om & true).sum()); or_all += int(om.sum())
    dev_frac, or_frac = dev_true / max(dev_all, 1), or_true / max(or_all, 1)
    print(f"{method}: winner inliers agreeing with the translation: device {dev_frac:.3f}, oracle {or_frac:.3f}")
    assert dev_all > 0 and dev_frac >= 0.95 * or_frac
