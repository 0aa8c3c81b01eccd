"""Pixels to verified matches for an unordered image set on the device (BASELINE configs[4] front end).

A photogrammetry capture is a set of photos of different sizes and orientations, each detected at its own size
(KeypointDetection.Detect takes a Matrix<Grayscale> of any dimensions).  The chain, with nothing read back but the
per-image keypoint counts:

    images -> pgm_detect_describe_images_batch_dev (one call for every image, optionally with the reference's NMS)
           -> compaction of each image's surviving descriptors and coordinates (one gather)
           -> the batch matcher over the pair list: "greedy" = pgm_match_pairs_batch_dev (upstream's MatchKeypoints),
              "ratio" = pgm_match_ratio_crosscheck_pairs_batch_dev (nearest / second nearest, ratio test, cross-check)
           -> pgm_ransac_fundamental_pairs_batch_dev (GetFundamentalMatrix of every pair)

This is the unordered-set counterpart of :func:`photogrammetry_b200.sequence.match_sequence_dev`.
"""
from __future__ import annotations

import time

import numpy as np

from ._lib import PGM_FLAG_PYTHON_GENERATION
from .sequence import pairs_table


class ImageSetResult:
    def __init__(self, counts, offsets, desc, xy, pair_list, matches, starts, match_counts, best, inliers, F, mask):
        self.counts = counts              # int32[K] keypoints per image
        self.offsets = offsets            # int64[K + 1] into desc / xy
        self.desc = desc                  # torch uint8[sum, stride] on the device
        self.xy = xy                      # torch int32[sum, 2]
        self.pair_list = pair_list        # int32[n_pairs, 2]
        self.matches = matches            # torch int32[3, total] (qi, tj, dist); pair p at starts[p] .. + match_counts[p]
        self.starts = starts              # int64[n_pairs]
        self.match_counts = match_counts  # int32[n_pairs]
        self.best = best                  # torch int32[n_pairs]: winning sample, -1 no inlier, -2 fewer matches than a sample
        self.inliers = inliers            # torch int32[n_pairs]
        self.F = F                        # torch float32[n_pairs, 3, 3]
        self.mask = mask                  # torch uint8[total]: inlier mask of each pair's winner, in the matches' slots


def match_image_set_dev(matcher, images, threshold: float, pairs: np.ndarray, *, nms_radius: int = -1, pair_list=None,
                        method: str = "greedy", ratio: float = 0.8, cross_check: bool = True, max_dist: int = -1,
                        n_samples: int = 2000, pairs_per_sample: int = 32, ransac_threshold: float = 0.001,
                        seed: int = 0, flags: int = 0, timings: dict | None = None) -> ImageSetResult:
    """``images``: list of 2-D torch float32 tensors on the matcher's GPU, any sizes (grey values on the generation's
    scale); ``pairs``: the BRIEF pair table; ``pair_list``: int32[n, 2] image pairs (default: all pairs a < b);
    ``flags``: 0 (the C# generation) or PGM_FLAG_PYTHON_GENERATION.  ``nms_radius >= 0`` matches the keypoints that
    survive the reference's NMS of that radius.  ``timings`` (optional) receives ms per stage."""
    import torch

    from .sharding import all_pairs
    if method not in ("greedy", "ratio"):
        raise ValueError(f"method must be 'greedy' or 'ratio', not {method!r}")
    if flags & ~PGM_FLAG_PYTHON_GENERATION:
        raise ValueError("flags: only PGM_FLAG_PYTHON_GENERATION is defined here")
    table = pairs_table(pairs)
    desc_bits = len(table)
    k = len(images)
    plist = all_pairs(k) if pair_list is None else np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
    dev = images[0].device if k else torch.device("cuda", matcher.device)
    stream = torch.cuda.current_stream(dev)
    py = bool(flags & PGM_FLAG_PYTHON_GENERATION)

    t0 = time.perf_counter()
    cap = 4096
    while True:                                  # a truncated image is detected again with room for all its keypoints
        xy, _sc, desc, counts = matcher.detect_describe_images_batch_dev(images, threshold, table, capacity=cap,
                                                                         python_generation=py, nms_radius=nms_radius)
        if not len(counts) or int(counts.max()) <= cap:
            break
        cap = int(counts.max())
    t1 = time.perf_counter()
    offs = np.zeros(k + 1, dtype=np.int64)
    offs[1:] = np.cumsum(counts)
    rows = np.concatenate([z * cap + np.arange(int(counts[z]), dtype=np.int64) for z in range(k)]) if k else np.zeros(0, np.int64)
    d_rows = torch.from_numpy(rows).to(dev, non_blocking=False)
    d_desc = desc.reshape(k * cap, -1).index_select(0, d_rows) if k else desc.reshape(0, desc.shape[-1])
    d_xy = xy.reshape(k * cap, 2).index_select(0, d_rows) if k else xy.reshape(0, 2)
    stream.synchronize()
    t2 = time.perf_counter()

    if method == "greedy":
        n1s = np.diff(offs)[plist[:, 0]] if len(plist) else np.zeros(0, np.int64)
        starts = np.concatenate([[0], np.cumsum(n1s)]).astype(np.int64)
        total = int(starts[-1])
        out = torch.empty((3, max(total, 1)), dtype=torch.int32, device=dev)
        with matcher.torch_ordered(dev):
            mcounts = matcher.match_pairs_batch_dev(d_desc.data_ptr(), offs, plist, desc_bits, int(d_desc.shape[1]),
                                                    out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), total)
        starts = starts[:-1]
    else:
        out, starts, mcounts = matcher.match_ratio_crosscheck_pairs_batch_dev(d_desc, offs, plist, desc_bits, ratio,
                                                                              cross_check, max_dist)
    stream.synchronize()
    t3 = time.perf_counter()

    best, inliers, F, mask = matcher.ransac_fundamental_pairs_batch_dev(
        d_xy, offs, plist, out[0], out[1], starts, mcounts, n_samples=n_samples, pairs_per_sample=pairs_per_sample,
        threshold=ransac_threshold, seed=seed)
    stream.synchronize()
    t4 = time.perf_counter()
    if timings is not None:
        timings.update({"detect_ms": (t1 - t0) * 1e3, "compaction_ms": (t2 - t1) * 1e3, "match_ms": (t3 - t2) * 1e3,
                        "ransac_ms": (t4 - t3) * 1e3})
    return ImageSetResult(counts, offs, d_desc, d_xy, plist, out, starts, mcounts, best, inliers, F, mask)
