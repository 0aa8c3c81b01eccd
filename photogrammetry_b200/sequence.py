"""Consecutive-frame matching of an image sequence on the device (BASELINE configs[2], SURVEY.md section 8d config 3).

The reference names a rendered Blender camera pan (blender/15pt_star_camera_pan) but ships only the .blend file; the
documented stand-in (SURVEY D5) is the construction of python_src/scripts/image_editing.py:8-15 -- the 15-point star
shifted right by a growing offset, columns shifted out of the frame dropped, vacated columns black -- here
K = 32 frames at 5 k px.  The pipeline is the reference's own chain (TestService.cs:80-96 per pair; FAST-12 + BRIEF of
the Python generation, which the reference tree can execute): detector -> descriptors -> matcher, all on the GPU:

    frames (one H2D) -> pgm_detect_describe_batch_dev (6 kernels for all frames, one read-back of K counts), or with
                        NMS pgm_detect_nms_describe_batch_dev (every NMS round on the device, one more read-back)
                     -> pgm_match_pairs_batch_dev over the K - 1 consecutive pairs (greedy, the reference's MatchKeypoints)
                     -> pgm_match_ratio_crosscheck_batch_dev: nearest / second nearest + ratio test + cross-check of every
                        consecutive pair in one launch (the north_star extension)
"""
from __future__ import annotations

import os
import time
from typing import List, Tuple

import numpy as np


def shifted_frames(gray: np.ndarray, n_frames: int = 32, step: int = 5) -> np.ndarray:
    """``[n_frames, H, W]``: frame k is ``gray`` shifted right by ``step * k`` pixels exactly as
    scripts/image_editing.py:8-15 does it (``new[row, col + offset] = image[row, col]`` for ``col < width - offset``)."""
    gray = np.asarray(gray)
    h, w = gray.shape
    out = np.zeros((n_frames, h, w), dtype=gray.dtype)
    for k in range(n_frames):
        off = step * k
        if off < w:
            out[k, :, off:] = gray[:, :w - off]
    return out


def star_gray() -> np.ndarray:
    """The committed grayscale of data/feature_matching_test/15pt_star.png (uint8[383, 451], tests/golden/star_detect.npz)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return np.load(os.path.join(root, "tests", "golden", "star_detect.npz"))["gray0"]


def star_pairs() -> np.ndarray:
    """The seeded Gaussian pair table the golden vectors were made with (int32[256, 4] = dx1, dy1, dx2, dy2 rows are built
    from the [256, 2, 2] (height, width) offsets of models/keypoint.py:52-57)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return np.load(os.path.join(root, "tests", "golden", "star_detect.npz"))["pairs"]


def pairs_table(pairs: np.ndarray) -> np.ndarray:
    """[n, 2, 2] (dy, dx) offset pairs of the Python generation -> int32[n, 4] (dx1, dy1, dx2, dy2)."""
    p = np.asarray(pairs)
    if p.ndim == 2 and p.shape[1] == 4:
        return np.ascontiguousarray(p, dtype=np.int32)
    return np.ascontiguousarray(np.stack([p[:, 0, 1], p[:, 0, 0], p[:, 1, 1], p[:, 1, 0]], axis=1), dtype=np.int32)


class SequenceResult:
    def __init__(self, counts, offsets, desc, xy, greedy, greedy_starts, greedy_counts, filtered):
        self.counts = counts                # int32[K] keypoints per frame
        self.offsets = offsets              # int64[K + 1] into desc / xy
        self.desc = desc                    # torch uint8[sum, stride] on the device
        self.xy = xy                        # torch int32[sum, 2]
        self.greedy = greedy                # torch int32[3, sum over pairs of n1] (qi, tj, dist), reference order per pair
        self.greedy_starts = greedy_starts  # int64[K - 1]
        self.greedy_counts = greedy_counts  # int32[K - 1]
        self.filtered = filtered            # list of torch int32[3, count_k]: ratio + cross-check survivors per pair


def match_sequence_dev(matcher, d_frames, threshold: float, pairs: np.ndarray, ratio: float = 0.8,
                       cross_check: bool = True, capacity: int = 4096, python_generation: bool = True,
                       desc_bits: int = 256, timings: dict | None = None, nms_radius: int = -1) -> SequenceResult:
    """``d_frames``: torch float32 ``[K, H, W]`` on the matcher's GPU (grey values on the generation's scale).
    ``nms_radius >= 0`` matches the keypoints that survive the reference's NMS (RedundantKeypointEliminator) of that
    radius, as the C# pipeline does (BuildKeypointDetectorPipeline, TestService.cs:94-95)."""
    import torch

    from .sharding import consecutive_pairs
    table = pairs_table(pairs)
    t0 = time.perf_counter()
    xy, _sc, desc, counts = matcher.detect_describe_batch_dev(d_frames, threshold, table, capacity=capacity,
                                                              python_generation=python_generation, nms_radius=nms_radius)
    if (counts > capacity).any():
        raise ValueError(f"a frame has {int(counts.max())} keypoints, more than capacity={capacity}")
    t1 = time.perf_counter()
    k = len(counts)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    d_desc = torch.cat([desc[f, :int(counts[f])] for f in range(k)]).contiguous()
    d_xy = torch.cat([xy[f, :int(counts[f])] for f in range(k)]).contiguous()
    plist = consecutive_pairs(k)
    n1s = counts[plist[:, 0]] if len(plist) else np.zeros(0, np.int64)
    starts = np.concatenate([[0], np.cumsum(n1s)]).astype(np.int64)
    total = int(starts[-1])
    out = torch.empty((3, max(total, 1)), dtype=torch.int32, device=d_frames.device)
    with matcher.torch_ordered(d_frames.device):
        gcounts = matcher.match_pairs_batch_dev(d_desc.data_ptr(), offs, plist, desc_bits, int(d_desc.shape[1]),
                                                out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), total)
    torch.cuda.current_stream(d_frames.device).synchronize()
    t2 = time.perf_counter()
    if len(plist):
        fo, fstarts, fcounts = matcher.match_ratio_crosscheck_batch_dev(d_desc, offs, plist, desc_bits, ratio, cross_check, -1)
        filtered = [fo[:, int(fstarts[k]):int(fstarts[k]) + int(fcounts[k])] for k in range(len(plist))]
    else:
        filtered = []
    torch.cuda.current_stream(d_frames.device).synchronize()
    t3 = time.perf_counter()
    if timings is not None:
        timings.update({"detect_describe_ms": (t1 - t0) * 1e3, "greedy_match_ms": (t2 - t1) * 1e3,
                        "ratio_crosscheck_ms": (t3 - t2) * 1e3})
    return SequenceResult(counts, offs, d_desc, d_xy, out[:, :total], starts[:-1], gcounts, filtered)


def bench_star_sequence(matcher, stream, dev, n_frames: int = 32, step: int = 5, reps: int = 5) -> dict:
    """ms per sequence and stage split of the configs[2] proxy (device resident after one upload of the frames)."""
    import torch
    frames = shifted_frames(star_gray(), n_frames, step).astype(np.float32)
    pairs = star_pairs()
    with torch.cuda.stream(stream):
        d_frames = torch.from_numpy(frames).to(dev)
        best, split, res = None, None, None
        for _ in range(reps + 1):
            tm = {}
            t0 = time.perf_counter()
            res = match_sequence_dev(matcher, d_frames, 50.0, pairs, timings=tm)
            dt = (time.perf_counter() - t0) * 1e3
            if best is None or dt < best:
                best, split = dt, tm
    evals = float(sum(int(res.counts[k]) * int(res.counts[k + 1]) for k in range(n_frames - 1)))
    return {"frames": n_frames, "shift_px_per_frame": step, "keypoints_per_frame": [int(x) for x in res.counts],
            "pairs": n_frames - 1, "ms_per_sequence": best, "stage_split_ms": split,
            "distance_evals": evals, "evals_per_s": evals / (best * 1e-3),
            "greedy_matches": int(sum(min(int(res.counts[k]), int(res.counts[k + 1])) for k in range(n_frames - 1))),
            "ratio_crosscheck_matches": int(sum(int(f.shape[1]) for f in res.filtered)),
            "note": "proxy for the un-rendered Blender pan (SURVEY D5): 15pt_star shifted 5 px per frame as "
                    "scripts/image_editing.py:8-15; FAST-12 threshold 50 + BRIEF-256 of the Python generation on the "
                    "device; greedy MatchKeypoints of all consecutive pairs in one batch call, ratio 0.8 + cross-check of all pairs in one launch"}
