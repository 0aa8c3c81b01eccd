"""pgm_detect_nms_describe_batch_dev: FAST-12 -> NMS -> BRIEF for a stack of device-resident images in one call, with
every NMS round on the device.  Per image the result must equal pgm_detect_describe_dev(nms_radius) bit for bit
(coordinates, FastScore, descriptor bytes, the reference's output order), and the oracle chain
(detect -> eliminate_redundant -> brief_descriptors) where it is cheap enough to run."""
import numpy as np
import pytest

from oracle import detect_np as D
from oracle import orc
from photogrammetry_b200 import keypoint_detection as kd
from photogrammetry_b200 import sequence, synthetic
from photogrammetry_b200._lib import PGM_E_INVALID_ARG, PGM_OK
from photogrammetry_b200.descriptors import pack_descriptors

pytestmark = pytest.mark.gpu

CS_PAIRS = D.gaussian_pairs(11, 256, 50)                 # (dx, dy) pairs of the C# generation, [256, 2, 2]
CS_TABLE = CS_PAIRS.reshape(-1, 4).astype(np.int32)
PY_TABLE = sequence.pairs_table(sequence.star_pairs())


def _star_frames(python_generation):
    """The 32 shifted-star frames on the generation's scale: 0..255 (Python) or Grayscale.K of the frame as RGB (C#)."""
    fr = sequence.shifted_frames(sequence.star_gray(), 32, 5)
    if python_generation:
        return fr.astype(np.float32)
    return np.stack([kd.grayscale_from_rgb8(np.repeat(f[..., None], 3, axis=2)) for f in fr])


def _random_frames():
    rng = np.random.default_rng(31)
    fr = rng.integers(0, 256, size=(6, 61, 83)).astype(np.float32)
    fr[3] = 77.0                                          # constant: no keypoint
    return fr


def _per_image(matcher, d_frames, th, table, r, pg):
    return [tuple(x.cpu().numpy() for x in matcher.detect_describe_dev(d_frames[k], th, table, nms_radius=r,
                                                                      python_generation=pg, capacity=65536))
            for k in range(d_frames.shape[0])]


def _assert_batch_equals(batch, per_image):
    xy, sc, desc, counts = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in batch)
    for k, (exy, esc, edesc) in enumerate(per_image):
        n = len(exy)
        assert int(counts[k]) == n, k
        assert (xy[k, :n] == exy).all() and (sc[k, :n] == esc).all() and (desc[k, :n] == edesc).all(), k


@pytest.mark.parametrize("r", [0, 1, 10, 200])
@pytest.mark.parametrize("pg", [False, True])
def test_random_frames_equal_per_image_calls(matcher, pg, r):
    import torch
    d = torch.from_numpy(_random_frames()).cuda()
    got = matcher.detect_describe_batch_dev(d, 40.0, CS_TABLE, capacity=4096, python_generation=pg, nms_radius=r)
    exp = _per_image(matcher, d, 40.0, CS_TABLE, r, pg)
    assert len(exp[3][0]) == 0 and sum(len(e[0]) for e in exp) > 0
    _assert_batch_equals(got, exp)


@pytest.mark.parametrize("r", [0, 1, 10, 200])
@pytest.mark.parametrize("pg", [False, True])
def test_star_frames_equal_per_image_calls(matcher, pg, r):
    import torch
    d = torch.from_numpy(_star_frames(pg)).cuda()
    th, table = (50.0, PY_TABLE) if pg else (0.1, CS_TABLE)
    got = matcher.detect_describe_batch_dev(d, th, table, capacity=4096, python_generation=pg, nms_radius=r)
    _assert_batch_equals(got, _per_image(matcher, d, th, table, r, pg))


def _oracle_chain(img, th, radius, pairs=CS_PAIRS):
    xy, sc = D.detect_vectorised(img, th)
    kept = D.eliminate_redundant_vectorised(xy, sc, radius)
    return xy[kept], sc[kept], pack_descriptors(D.brief_descriptors(img, xy[kept], pairs), 256), len(xy)


def test_star_frames_equal_oracle_chain(matcher):
    import torch
    frames = _star_frames(False)
    xy, sc, desc, counts = matcher.detect_describe_batch_dev(torch.from_numpy(frames).cuda(), 0.1, CS_TABLE, nms_radius=10)
    xy, sc, desc = xy.cpu().numpy(), sc.cpu().numpy(), desc.cpu().numpy()
    for k in range(32):
        f_xy, f_sc = D.detect_vectorised(frames[k], 0.1)
        kept = D.eliminate_redundant(f_xy, f_sc, 10)
        exp_desc = pack_descriptors(D.brief_descriptors(frames[k], f_xy[kept], CS_PAIRS), 256)
        n = len(kept)
        assert counts[k] == n and (xy[k, :n] == f_xy[kept]).all() and (sc[k, :n] == f_sc[kept]).all(), k
        assert (desc[k, :n] == exp_desc).all(), k
        if k in (0, 15, 31):
            assert (len(f_xy), n) == {0: (126, 30), 15: (123, 29), 31: (99, 23)}[k]


def test_chain_frame_one_sync(matcher):
    """The dotted row needs 496 parallel rounds (each decides one dot); the call still synchronises once."""
    import torch
    rng = np.random.default_rng(4)
    frames = np.stack([synthetic.dotted_row_image(), rng.random((40, 2000), dtype=np.float32),
                       np.zeros((40, 2000), np.float32)])
    xy, sc, desc, d_counts = matcher.detect_describe_batch_dev(torch.from_numpy(frames).cuda(), 0.1, CS_TABLE,
                                                               read_counts=False, nms_radius=4)
    st = matcher.stats()
    counts = d_counts.cpu().numpy()
    assert st["host_syncs"] == 1
    assert counts[0] == 248 and counts[2] == 0
    for k in range(2):
        exy, esc, edesc, n_fast = _oracle_chain(frames[k], 0.1, 4)
        if k == 0:
            assert n_fast == 496 and (exy[:, 0] == np.arange(8, 1989, 8)).all()
        n = len(exy)
        assert counts[k] == n
        assert (xy[k, :n].cpu().numpy() == exy).all() and (sc[k, :n].cpu().numpy() == esc).all()
        assert (desc[k, :n].cpu().numpy() == edesc).all()


def test_large_frames(matcher):
    import torch
    frames = np.stack([synthetic.rectangles_image(), synthetic.rectangles_image(shift=150)])
    d = torch.from_numpy(frames).cuda()
    got = matcher.detect_describe_batch_dev(d, 0.1, CS_TABLE, capacity=8192, nms_radius=10)
    assert matcher.stats()["host_syncs"] == 2
    _assert_batch_equals(got, _per_image(matcher, d, 0.1, CS_TABLE, 10, False))
    f_xy, f_sc = D.detect_vectorised(frames[0], 0.1)
    kept = D.eliminate_redundant_vectorised(f_xy, f_sc, 10)
    assert (len(f_xy), len(kept)) == (58196, 6233)
    assert int(got[3][0]) == 6233 and (got[0][0, :6233].cpu().numpy() == f_xy[kept]).all()


# ---- the C ABI directly: caller-owned outputs, refusals ------------------------------------------------------------
SENTINEL = -7


def _call(matcher, d_frames, th, r, cap, table=CS_TABLE, read_counts=True, n_images=None, width=None, stride=32):
    """The C# generation through the C ABI into outputs pre-filled with a sentinel, one image's slots more than needed."""
    import torch
    k, hgt, wid = (int(x) for x in d_frames.shape)
    dev = d_frames.device
    out = (torch.full((k + 1, max(cap, 1), 2), SENTINEL, dtype=torch.int32, device=dev),
           torch.full((k + 1, max(cap, 1)), SENTINEL, dtype=torch.int32, device=dev),
           torch.full((k + 1, max(cap, 1), stride), 0xA5, dtype=torch.uint8, device=dev),
           torch.full((k + 1,), SENTINEL, dtype=torch.int32, device=dev))
    h_cnt = np.full(k + 1, SENTINEL, dtype=np.int32)
    with matcher.torch_ordered(dev):
        rc = matcher._lib.pgm_detect_nms_describe_batch_dev(
            matcher._h, d_frames.data_ptr(), k if n_images is None else n_images, wid if width is None else width, hgt,
            float(th), int(r), table.ctypes.data, len(table), stride, 0, out[0].data_ptr(), out[1].data_ptr(),
            out[2].data_ptr(), cap, out[3].data_ptr(), h_cnt.ctypes.data if read_counts else None)
    return rc, out, h_cnt


def test_truncation(matcher):
    import torch
    d = torch.from_numpy(_star_frames(False)[12:28]).cuda()            # 30 down to 25 survivors
    k_img = int(d.shape[0])
    full = matcher.detect_describe_batch_dev(d, 0.1, CS_TABLE, capacity=4096, nms_radius=10)
    counts = full[3]
    cap = 27
    assert counts.min() < cap < counts.max()
    for read_counts in (True, False):
        rc, (xy, sc, desc, d_cnt), h_cnt = _call(matcher, d, 0.1, 10, cap, read_counts=read_counts)
        assert rc == PGM_OK
        xy, sc, desc, d_cnt = (x.cpu().numpy() for x in (xy, sc, desc, d_cnt))
        assert (d_cnt[:k_img] == counts).all() and d_cnt[k_img] == SENTINEL
        if read_counts:
            assert (h_cnt[:k_img] == counts).all()
        for k in range(k_img):
            m = min(int(counts[k]), cap)
            assert (xy[k, :m] == full[0][k, :m].cpu().numpy()).all() and (sc[k, :m] == full[1][k, :m].cpu().numpy()).all()
            assert (desc[k, :m] == full[2][k, :m].cpu().numpy()).all()
            assert (xy[k, m:] == SENTINEL).all() and (sc[k, m:] == SENTINEL).all() and (desc[k, m:] == 0xA5).all()
        assert (xy[k_img] == SENTINEL).all() and (sc[k_img] == SENTINEL).all() and (desc[k_img] == 0xA5).all()


def test_refusals_and_empty_batch(matcher):
    import torch
    d = torch.from_numpy(_random_frames()).cuda()
    assert _call(matcher, d, 40.0, -1, 64)[0] == PGM_E_INVALID_ARG
    assert _call(matcher, d, 40.0, 10, 0)[0] == PGM_E_INVALID_ARG              # capacity < 1
    assert _call(matcher, d, 40.0, 10, 64, n_images=-1)[0] == PGM_E_INVALID_ARG
    assert _call(matcher, d, 40.0, 10, 64, width=0)[0] == PGM_E_INVALID_ARG
    assert _call(matcher, d, 40.0, 10, 64, width=70000)[0] == PGM_E_INVALID_ARG
    assert _call(matcher, d, 40.0, 10, 64, stride=24)[0] == PGM_E_INVALID_ARG       # not a multiple of 16
    assert _call(matcher, d, 40.0, 10, 64, stride=16)[0] == PGM_E_INVALID_ARG       # 256 pairs need 32 bytes
    assert matcher._lib.pgm_detect_nms_describe_batch_dev(
        matcher._h, None, 6, 83, 61, 40.0, 10, CS_TABLE.ctypes.data, 256, 32, 0, None, None, None, 64, None,
        None) == PGM_E_INVALID_ARG
    rc, out, h_cnt = _call(matcher, d, 40.0, 10, 64, n_images=0)
    assert rc == PGM_OK and (h_cnt == SENTINEL).all() and (out[3].cpu().numpy() == SENTINEL).all()
    assert (out[0].cpu().numpy() == SENTINEL).all()
    st = matcher.stats()
    assert st["host_syncs"] == 0 and st["kernel_launches"] == 0


def test_launches_independent_of_rounds_and_images(matcher):
    import torch
    launches = []
    for frames, r in ((synthetic.dotted_row_image()[None], 4), (np.repeat(synthetic.dotted_row_image()[None], 5, 0), 4),
                      (np.repeat(synthetic.dotted_row_image()[None], 5, 0), 0)):
        matcher.detect_describe_batch_dev(torch.from_numpy(frames).cuda(), 0.1, CS_TABLE, nms_radius=r)
        launches.append(matcher.stats()["kernel_launches"])
    assert len(set(launches)) == 1


def test_non_default_stream(matcher):
    import torch
    frames = _star_frames(True)
    ref = matcher.detect_describe_batch_dev(torch.from_numpy(frames).cuda(), 50.0, PY_TABLE, python_generation=True,
                                            nms_radius=10)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d = torch.from_numpy(frames).cuda()
        got = matcher.detect_describe_batch_dev(d, 50.0, PY_TABLE, python_generation=True, nms_radius=10,
                                                read_counts=False)
        got = [x.cpu().numpy() for x in got]
    assert (got[3] == ref[3]).all()
    for k, n in enumerate(ref[3]):                # (slots past an image's count are never written)
        for g, r in zip(got[:3], ref[:3]):
            assert (g[k, :n] == r[k, :n].cpu().numpy()).all(), k


def test_sequence_chain_with_nms(matcher):
    """The C# generation's chain for the whole star sequence: Detect -> NMS -> BRIEF -> MatchKeypoints, then the ratio
    test and cross-check, every consecutive pair against the oracle."""
    import torch
    frames = _star_frames(False)
    res = sequence.match_sequence_dev(matcher, torch.from_numpy(frames).cuda(), 0.1, CS_TABLE, nms_radius=10,
                                      python_generation=False)
    descs = []
    for k in range(32):
        exy, _esc, edesc, _ = _oracle_chain(frames[k], 0.1, 10)
        assert int(res.counts[k]) == len(exy)
        assert (res.xy[res.offsets[k]:res.offsets[k + 1]].cpu().numpy() == exy).all()
        assert (res.desc[res.offsets[k]:res.offsets[k + 1]].cpu().numpy() == edesc).all()
        descs.append(edesc)
    greedy = res.greedy.cpu().numpy()
    for k in range(31):
        q, t = descs[k], descs[k + 1]
        exp = orc.match_sweep(q, t)
        got = greedy[:, res.greedy_starts[k]:res.greedy_starts[k] + res.greedy_counts[k]].T
        assert got.shape == exp.shape and (got == exp).all(), k
        expf = orc.match_ratio_crosscheck(q, t, 0.8, True)
        gotf = res.filtered[k].cpu().numpy().T
        assert gotf.shape == expf.shape and (gotf == expf).all(), k
