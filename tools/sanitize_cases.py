"""The small cases run under compute-sanitizer (memcheck / racecheck / synccheck / initcheck, one tool per gpurun call):

    compute-sanitizer --tool memcheck python tools/sanitize_cases.py

  1. 1024 x 1024 single pair: latency mode -- init, round 0, the persistent tail kernel with its hand-rolled grid barrier,
     candidate-edge filter, sparse sub-rounds, finisher_prepare -> finisher hand-over through global memory, sliced ordering
  2. 300 x 280 all-duplicate descriptors: every distance is 0 (candidate lists overflow, one accept per round, n1 > n2 tail)
  3. 24 pairs of 512 x 512: throughput mode (standalone round / accept+filter / sparse / finisher / order kernels)
  4. float L2 512 x 512, D = 128: the tcgen05 CTA-pair kernel with its cluster mbarriers
  5. 3 emulated train shards of a 700 x 650 pair (export / propose / stable commit kernels)
  6. ratio test + cross-check of 7 pairs of any size, empty and split ones included (fused distance pass with
     column splits, split-partial merge, block-parallel ordered compaction)
  7. float L2 batch of 6 pairs: one large pair whose row pairs span several segments (split candidate slots), flagged
     rows in two pairs (crowded band, identical train rows) taken by the batched fallback, then the ratio + cross-check
     filter with its reversed pairs and ordered compaction
  8. batched fundamental-matrix RANSAC of 6 pairs: one below P, a degenerate one (every keypoint the same pixel), one of
     20 000 matches (several shared-memory tiles per score CTA), S spread over two score items per pair
  9. batched detect -> NMS -> BRIEF of 4 frames: the dotted-row chain (496 device-side rounds in the cooperative kernel),
     a blank frame (empty run) and two random frames, against the oracle chain
 10. detect -> NMS -> BRIEF of a set of images of different sizes in one call (flat FAST tiles and row slots,
     per-image NMS cells): landscape and portrait frames, odd widths, a 5 x 9 image with no FAST interior and the
     dotted-row chain, with gaps between the images, against single-image calls
Every result is checked against the oracle, so a sanitizer run is also a parity run."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from oracle import orc
from photogrammetry_b200 import sharding, synthetic
from photogrammetry_b200.keypoint_matching import Matcher

m = Matcher(0)
q, t = synthetic.config2_pair(1024, "U")
assert (m.match_greedy(q, t, 256) == orc.match_sweep(q, t)).all()
print("case 1 ok", m.stats())
d = np.tile(synthetic.uniform_descriptors(3, 1, 256), (300, 1))
assert (m.match_greedy(d, d[:280], 256) == orc.match_sweep(d, d[:280])).all()
print("case 2 ok")
per, n_img = 512, 9
imgs = np.concatenate([synthetic.uniform_descriptors(100 + k, per, 256) for k in range(n_img)])
offs = np.arange(n_img + 1, dtype=np.int64) * per
pairs = sharding.all_pairs(n_img)[:24]
tr, starts, counts = m.match_pairs_batch(imgs, offs, pairs, 256)
for p, (a, b) in enumerate(pairs):
    assert (tr[starts[p]:starts[p] + counts[p]] == orc.match_sweep(imgs[offs[a]:offs[a + 1]], imgs[offs[b]:offs[b + 1]])).all()
print("case 3 ok", m.stats())
rng = np.random.default_rng(1)
fq, ft = rng.random((512, 128), dtype=np.float32), rng.random((512, 128), dtype=np.float32)
bj, bd, sj, sd = m.knn2_l2(fq, ft)
ej, ed, _, _ = orc.l2_knn2(fq, ft)
assert (np.abs(bd - ed) <= 1e-4 * np.maximum(ed, 1e-12)).all() and (bj != ej).mean() <= 0.01
print("case 4 ok")
q, t = synthetic.uniform_descriptors(5, 700, 256), synthetic.uniform_descriptors(6, 650, 256)
outs, rounds = sharding.match_train_sharded_emulated(m, q, t, 3)
exp = orc.match_sweep(q, t)
assert all((o == exp).all() for o in outs)
print("case 5 ok", rounds)
sizes = [0, 1, 700, 2600, 900]
base = synthetic.uniform_descriptors(7, max(sizes), 256)
imgs = [base[:n] if k % 2 == 0 else synthetic.noisy_copy_descriptors(8 + k, base, 256)[:n] for k, n in enumerate(sizes)]
offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
pairs = [(2, 3), (3, 2), (3, 4), (4, 4), (1, 3), (3, 1), (0, 2), (2, 0)]
d_all = torch.from_numpy(np.concatenate(imgs)).cuda()
for ratio, cc, md in [(0.8, True, -1), (0.0, False, 60)]:
    out, starts, counts = m.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, 256, ratio, cc, md)
    out = out.cpu().numpy()
    for p, (a, b) in enumerate(pairs):
        assert (out[:, starts[p]:starts[p] + counts[p]].T == orc.match_ratio_crosscheck(imgs[a], imgs[b], ratio, cc, md)).all()
print("case 6 ok", m.stats())
rng = np.random.default_rng(9)
big_q, big_t = rng.random((2600, 128), dtype=np.float32), rng.random((9000, 128), dtype=np.float32)
crowd_q, crowd_t = rng.standard_normal((600, 128)).astype(np.float32), rng.standard_normal((3000, 128)).astype(np.float32)
for k in range(12):
    crowd_t[100 + k] = crowd_q[7] + np.float32(0.01 * (12 - k)) * np.eye(128, dtype=np.float32)[3]
same_q, same_t = rng.standard_normal((300, 128)).astype(np.float32), np.tile(rng.standard_normal((1, 128)).astype(np.float32), (5000, 1))
imgs = [big_q, big_t, crowd_q, crowd_t, same_q, same_t, rng.standard_normal((100, 128)).astype(np.float32)]
offs = np.concatenate([[0], np.cumsum([len(x) for x in imgs])]).astype(np.int64)
pairs = np.array([(0, 1), (2, 3), (4, 5), (6, 2), (3, 2), (1, 0)], dtype=np.int32)
d_all = torch.from_numpy(np.concatenate(imgs)).cuda()
res = [x.cpu().numpy() for x in m.knn2_l2_pairs_batch_dev(d_all, offs, pairs)[:4]]
assert m.l2_last_fallback_rows() >= 301
rev = [x.cpu().numpy() for x in m.knn2_l2_pairs_batch_dev(d_all, offs, pairs[:, ::-1].copy())[:4]]
qi, tj, dist, starts, counts = (x.cpu().numpy() if hasattr(x, "cpu") else x
                                for x in m.match_l2_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, 0.8, True))
o = ro = 0
for p, (a, b) in enumerate(pairs):
    n1, n2 = len(imgs[a]), len(imgs[b])
    bj, bd, sj, sd = (x[o:o + n1] for x in res)
    ej, ed, fj, fd = orc.l2_knn2(imgs[a], imgs[b])
    for g_d, e_d in ((bd, ed), (sd, fd)):
        assert (np.abs(g_d - e_d) <= 1e-4 * np.maximum(e_d, 1e-12) + 1e-6).all()
    assert (bj != ej).mean() <= 0.01
    keep = (bd < np.float32(np.float32(0.8) * np.float32(0.8)) * sd) & (rev[0][ro:ro + n2][bj] == np.arange(n1))
    assert counts[p] == keep.sum() and (qi[starts[p]:starts[p] + counts[p]] == np.nonzero(keep)[0]).all()
    assert (tj[starts[p]:starts[p] + counts[p]] == bj[keep]).all() and (dist[starts[p]:starts[p] + counts[p]] == bd[keep]).all()
    o += n1; ro += n2
print("case 7 ok", m.stats())
from oracle import ransac_batch_np as R
xy, offs, pl, qi, tj, st, cn = synthetic.two_view_matches(11, 4, 400)
big = synthetic.two_view_matches(12, 1, 20000)
n_img = len(offs) - 1
xy = np.concatenate([xy, big[0], np.full((60, 2), (321, 654), np.int32)])
offs = np.concatenate([offs, offs[-1] + big[1][1:], [offs[-1] + big[1][-1] + 60]]).astype(np.int64)
pl = np.concatenate([pl, big[2] + n_img, [[n_img + 2, n_img + 2]]]).astype(np.int32)
qi = np.concatenate([qi, big[3], np.arange(60, dtype=np.int32)])
tj = np.concatenate([tj, big[4], np.arange(60, dtype=np.int32)])
st = np.concatenate([st, [len(st) * 400], [len(st) * 400 + 20000]]).astype(np.int64)
cn = np.concatenate([cn, [20000], [60]]).astype(np.int32)
cn[1] = 31                                                  # below P
d_xy, d_qi, d_tj = (torch.from_numpy(x).cuda() for x in (xy, qi, tj))
best, inl, F, mask = (x.cpu().numpy() for x in m.ransac_fundamental_pairs_batch_dev(
    d_xy, offs, pl, d_qi, d_tj, st, cn, n_samples=200, pairs_per_sample=32, threshold=0.001, seed=4, require_rank2=False))
exp = R.get_fundamental_pairs(xy, offs, pl, qi, tj, st, cn, 200, 32, 0.001, 4, require_rank2=False)
for p, (eb, ei, eF, em, _, _) in enumerate(exp):
    assert best[p] == eb and inl[p] == ei and (mask[st[p]:st[p] + cn[p]] == em).all(), p
    assert np.abs(F[p].astype(np.float64) - eF).max() <= 1e-6 * max(np.abs(eF).max(), 1e-30), p
assert best[1] == -2 and np.isfinite(F).all()
print("case 8 ok", m.stats())
from oracle import detect_np as D
from photogrammetry_b200.descriptors import pack_descriptors
rng = np.random.default_rng(12)
frames = np.stack([synthetic.dotted_row_image(), np.zeros((40, 2000), np.float32),
                   rng.random((40, 2000), dtype=np.float32), rng.random((40, 2000), dtype=np.float32)])
dpairs = D.gaussian_pairs(11, 256, 50)
xy, sc, desc, counts = m.detect_describe_batch_dev(torch.from_numpy(frames).cuda(), 0.1, dpairs.reshape(-1, 4),
                                                   capacity=4096, nms_radius=4)
for k in range(4):
    exy, esc = D.detect_vectorised(frames[k], 0.1)
    kept = D.eliminate_redundant_vectorised(exy, esc, 4)
    n = len(kept)
    assert counts[k] == n and (xy[k, :n].cpu().numpy() == exy[kept]).all() and (sc[k, :n].cpu().numpy() == esc[kept]).all()
    assert (desc[k, :n].cpu().numpy() == pack_descriptors(D.brief_descriptors(frames[k], exy[kept], dpairs), 256)).all()
assert counts[0] == 248 and counts[1] == 0
print("case 9 ok", m.stats())
ims = [rng.random((61, 83), dtype=np.float32), rng.random((83, 61), dtype=np.float32), rng.random((9, 5), dtype=np.float32),
       synthetic.dotted_row_image(), rng.random((33, 257), dtype=np.float32)]
buf, offs = [], [0]
for im in ims:                                               # 13 NaN pixels after every image
    buf += [im.ravel(), np.full(13, np.nan, np.float32)]
    offs.append(offs[-1] + im.size + 13)
d_buf = torch.from_numpy(np.concatenate(buf)).cuda()
views = [d_buf[offs[k]:offs[k] + im.size].view(im.shape) for k, im in enumerate(ims)]
xy, sc, desc, counts = m.detect_describe_images_batch_dev(views, 0.1, dpairs.reshape(-1, 4), capacity=4096, nms_radius=4)
for k, v in enumerate(views):
    exy, esc, edesc = (x.cpu().numpy() for x in m.detect_describe_dev(v.contiguous(), 0.1, dpairs.reshape(-1, 4), nms_radius=4))
    n = len(exy)
    assert counts[k] == n and (xy[k, :n].cpu().numpy() == exy).all() and (sc[k, :n].cpu().numpy() == esc).all(), k
    assert (desc[k, :n].cpu().numpy() == edesc).all(), k
assert counts[2] == 0 and counts[3] == 248
print("case 10 ok", m.stats())
m.close()
print("ALL OK")
