"""Seeded synthetic descriptor sets for the BASELINE configs (SURVEY.md section 8d).

A counter-based splitmix64 stream: the idx-th output of stream ``seed`` is
``mix(seed + (idx+1)*GAMMA)``, so the generator vectorises in numpy; the test
suite cross-checks it bit-for-bit against an independent C implementation of
the same stream.

Distributions:
  U  i.i.d. uniform W-bit descriptors.
  C  "noisy copy": train = permuted copy of query, each bit flipped with
     probability floor(256*flip_p)/256, then a fraction outlier_p of the rows
     replaced by uniform noise.
"""
from __future__ import annotations

import numpy as np

from .descriptors import stride_for_bits

_GAMMA = np.uint64(0x9E3779B97F4A7C15)
_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)


def _mix(z: np.ndarray) -> np.ndarray:
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
        return z ^ (z >> np.uint64(31))


def _sm64(seed: int, idx: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        return _mix(np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + (np.asarray(idx, dtype=np.uint64) + np.uint64(1)) * _GAMMA)


def _derive(seed: int, k: int) -> int:
    with np.errstate(over="ignore"):
        return int(_mix(np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + np.uint64(k) * _GAMMA))


def uniform_descriptors(seed: int, n: int, desc_bits: int = 256, stride: int | None = None) -> np.ndarray:
    """``uint8[n, stride]`` i.i.d. uniform ``desc_bits``-bit descriptors."""
    stride = stride or stride_for_bits(desc_bits)
    nw = (desc_bits + 63) // 64
    idx = np.arange(n * nw, dtype=np.uint64)
    words = _sm64(seed, idx).reshape(n, nw)
    top = desc_bits - 64 * (nw - 1)
    if top < 64:
        words[:, nw - 1] &= np.uint64((1 << top) - 1)
    out = np.zeros((n, stride), dtype=np.uint8)
    raw = words.astype("<u8").view(np.uint8).reshape(n, nw * 8)
    out[:, :min(stride, nw * 8)] = raw[:, :min(stride, nw * 8)]
    return out


def noisy_copy_descriptors(seed: int, query: np.ndarray, desc_bits: int = 256,
                           flip_p: float = 0.10, outlier_p: float = 0.30) -> np.ndarray:
    """Distribution C: permuted, bit-flipped copy of ``query`` with outlier rows."""
    query = np.ascontiguousarray(query, dtype=np.uint8)
    n, stride = query.shape
    s_perm, s_flip, s_out, s_noise = (_derive(seed, k) for k in (1, 2, 3, 4))
    rows = np.arange(n, dtype=np.uint64)
    perm = np.argsort(_sm64(s_perm, rows), kind="stable")
    out = query[perm].copy()
    nbytes = (desc_bits + 7) // 8
    thr = int(flip_p * 256.0)
    chunk = max(1, (1 << 22) // max(nbytes, 1))
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        idx = (np.arange(r0, r1, dtype=np.uint64)[:, None] * np.uint64(nbytes)
               + np.arange(nbytes, dtype=np.uint64)[None, :])
        draws = _sm64(s_flip, idx).astype("<u8").view(np.uint8).reshape(r1 - r0, nbytes, 8)
        bits = (draws < thr)
        bitpos = np.arange(nbytes)[:, None] * 8 + np.arange(8)[None, :]
        bits &= (bitpos < desc_bits)[None, :, :]
        mask = (bits.astype(np.uint8) << np.arange(8, dtype=np.uint8)[None, None, :]).sum(axis=2).astype(np.uint8)
        out[r0:r1, :nbytes] ^= mask
    u = (_sm64(s_out, rows) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    outlier = u < outlier_p
    if outlier.any():
        noise = uniform_descriptors(s_noise, n, desc_bits, stride)
        out[outlier] = noise[outlier]
    return out


def config2_pair(n: int = 8192, dist: str = "U", desc_bits: int = 256):
    """BASELINE configs[1]: one synthetic pair (query, train)."""
    if dist == "U":
        return uniform_descriptors(1234, n, desc_bits), uniform_descriptors(5678, n, desc_bits)
    if dist == "C":
        q = uniform_descriptors(1234, n, desc_bits)
        return q, noisy_copy_descriptors(42, q, desc_bits)
    raise ValueError(f"unknown distribution {dist!r}")


def two_view_matches(seed: int, n_pairs: int, per_pair: int = 512, outlier_frac: float = 0.3, size: int = 4000):
    """Match lists for the batched fundamental-matrix RANSAC: pair k = images (2k, 2k + 1), each with ``per_pair``
    keypoints that are projections of one set of 3D points by two pinhole cameras (focal length ``size / 2``, principal
    point at the image centre, second camera rotated by up to 0.1 rad and translated), rounded to pixels and clipped to
    ``[0, size)``.  Match i joins keypoint i of image 2k with the same point's keypoint of image 2k + 1 (stored in a
    permuted row order); a fraction ``outlier_frac`` of the matches points at a random keypoint instead.

    Returns ``(xy int32[2 n_pairs per_pair, 2], image_offsets int64, pair_list int32[n_pairs, 2], qi int32, tj int32,
    starts int64[n_pairs], counts int32[n_pairs])``: the layout the batch matchers produce."""
    rng = np.random.default_rng(seed)
    m = int(per_pair)
    X = np.stack([rng.uniform(-1, 1, (n_pairs, m)), rng.uniform(-1, 1, (n_pairs, m)), rng.uniform(4, 8, (n_pairs, m))], -1)
    ang = rng.uniform(-0.1, 0.1, (n_pairs, 3))
    cx, sx = np.cos(ang[:, 0]), np.sin(ang[:, 0])
    cy, sy = np.cos(ang[:, 1]), np.sin(ang[:, 1])
    cz, sz = np.cos(ang[:, 2]), np.sin(ang[:, 2])
    one, zero = np.ones(n_pairs), np.zeros(n_pairs)
    Rx = np.stack([one, zero, zero, zero, cx, -sx, zero, sx, cx], -1).reshape(-1, 3, 3)
    Ry = np.stack([cy, zero, sy, zero, one, zero, -sy, zero, cy], -1).reshape(-1, 3, 3)
    Rz = np.stack([cz, -sz, zero, sz, cz, zero, zero, zero, one], -1).reshape(-1, 3, 3)
    R = Rz @ Ry @ Rx
    t = rng.uniform(-0.5, 0.5, (n_pairs, 1, 3))
    f, c = size / 2.0, size / 2.0

    def project(P):
        return np.clip(np.rint(f * P[..., :2] / P[..., 2:3] + c), 0, size - 1).astype(np.int32)
    x1 = project(X)
    x2 = project(np.einsum("kij,kmj->kmi", R, X) + t)
    perm = rng.permuted(np.tile(np.arange(m), (n_pairs, 1)), axis=1)          # row of point i in image 2k + 1
    img2 = np.empty_like(x2)
    np.put_along_axis(img2, perm[..., None], x2, axis=1)
    tj = perm.copy()
    out = rng.random((n_pairs, m)) < outlier_frac
    tj[out] = rng.integers(0, m, size=int(out.sum()))
    xy = np.stack([x1, img2], axis=1).reshape(-1, 2)
    offs = np.arange(2 * n_pairs + 1, dtype=np.int64) * m
    pairs = np.stack([np.arange(n_pairs) * 2, np.arange(n_pairs) * 2 + 1], -1).astype(np.int32)
    qi = np.tile(np.arange(m, dtype=np.int32), n_pairs)
    return (np.ascontiguousarray(xy), offs, pairs, qi, tj.reshape(-1).astype(np.int32),
            np.arange(n_pairs, dtype=np.int64) * m, np.full(n_pairs, m, dtype=np.int32))


# ---- images for the keypoint producer -----------------------------------------------------------------------------
def rectangles_image(h: int = 3000, w: int = 4000, seed: int = 7, shift: int = 0) -> np.ndarray:
    """float32[h, w] on the Grayscale.K scale: 1500 random overlapping rectangles on 0.5 and 8000 random 3 x 3 blobs
    (tools/detect_one.py's image; 4000 x 3000 is the size of the reference's lego photographs), shifted right by
    ``shift`` px with the vacated columns black, as scripts/image_editing.py:8-15 shifts its frames."""
    rng = np.random.default_rng(seed)
    img = np.full((h, w), 0.5, dtype=np.float32)
    for _ in range(1500):
        x0, y0 = int(rng.integers(0, w - 40)), int(rng.integers(0, h - 40))
        rw, rh = int(rng.integers(20, 400)), int(rng.integers(20, 400))
        img[y0:y0 + rh, x0:x0 + rw] = np.float32(rng.random())
    for _ in range(8000):                      # small blobs: every ring pixel differs from the centre
        x0, y0 = int(rng.integers(5, w - 8)), int(rng.integers(5, h - 8))
        img[y0:y0 + 3, x0:x0 + 3] = np.float32(rng.random())
    if shift:
        out = np.zeros_like(img)
        out[:, shift:] = img[:, :w - shift]
        img = out
    return img


def dotted_row_image(h: int = 40, w: int = 2000, value: float = 1.0) -> np.ndarray:
    """float32[h, w], black but for a dot of ``value`` every 4 px on row 20 (x = 8, 12, ..., 1988 at the default
    size): 496 FAST keypoints of score 16 at threshold 0.1 (``value`` 255 and threshold 50 for the Python generation).
    At NMS radius 4 each dot suppresses its right neighbour only once it is itself kept, so the parallel rounds form a
    chain of 496 and every other dot survives (248)."""
    img = np.zeros((h, w), dtype=np.float32)
    img[20, 8:w - 8:4] = np.float32(value)
    return img


def scene_crops(seed: int, boxes):
    """Crops of one seeded scene (a :func:`rectangles_image` just large enough to hold every box): ``boxes`` is a list of
    ``(x0, y0, w, h)`` in scene pixels, so a set can mix sizes and portrait / landscape orientations.  Returns
    ``(crops, offsets)``: float32[h, w] copies and int64[len(boxes), 2] = (x0, y0).  A scene point at (x, y) in crop a
    is at (x + x0_a - x0_b, y + y0_a - y0_b) in crop b: overlapping crops are a pure translation apart, which gives
    their correspondences a known ground truth."""
    boxes = np.asarray(boxes, dtype=np.int64).reshape(-1, 4)
    if (boxes[:, :2] < 0).any() or (boxes[:, 2:] < 1).any():
        raise ValueError("boxes need x0, y0 >= 0 and w, h >= 1")
    w = max(int((boxes[:, 0] + boxes[:, 2]).max()), 64)
    h = max(int((boxes[:, 1] + boxes[:, 3]).max()), 64)
    scene = rectangles_image(h, w, seed)
    crops = [np.ascontiguousarray(scene[y0:y0 + bh, x0:x0 + bw]) for x0, y0, bw, bh in boxes.tolist()]
    return crops, np.ascontiguousarray(boxes[:, :2])
