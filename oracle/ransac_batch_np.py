"""numpy oracle of the batched fundamental-matrix RANSAC (pgm_ransac_fundamental_pairs_batch_dev) -- TEST
INFRASTRUCTURE ONLY.

  CameraPoseEstimation.GetFundamentalMatrix       dotnet_src/ImageProcessing/CameraPoseEstimation.cs:26-94
  CameraPoseEstimation.EstimateFundamentalMatrix  :204-250, CalculateTransformationMatrix :252-275

The per-sample work the host mirror (photogrammetry_b200/camera_pose_estimation.py) restates -- translation-only
normalised 8-point estimate, rank gate -- with the library's seeded sampler in place of upstream's unseeded
``OrderBy(random)`` (parity with the reference is statistical only).  The null vector comes from numpy's fp64 SVD of A;
scoring is ``ransac_np.score``, unchanged.
"""
from __future__ import annotations

import numpy as np

from .ransac_np import score

_M64 = (1 << 64) - 1


def _splitmix64(z: int) -> int:
    z = (z + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def sample_indices(count: int, P: int, seed: int, a: int, b: int, s: int) -> np.ndarray:
    """int64[P]: the P distinct indices in [0, count) hypothesis s of image pair (a, b) draws (Floyd's algorithm on the
    counter-based splitmix64 draws include/pgmatch.h states), ascending."""
    count, P, seed, a, b, s = (int(x) for x in (count, P, seed, a, b, s))
    key = _splitmix64((seed & _M64) ^ _splitmix64(((a & 0xFFFFFFFF) << 32) | (b & 0xFFFFFFFF)))
    chosen = set()
    for t in range(P):
        j = count - P + t
        u = _splitmix64(key ^ (((s & 0xFFFFFFFF) << 32) | t)) >> 32
        r = (u * (j + 1)) >> 32
        chosen.add(j if r in chosen else r)
    return np.array(sorted(chosen), dtype=np.int64)


def design_matrix(xy1, xy2):
    """(A float32[..., P, 9], T1, T2 float64[..., 3, 3]) of the translation-only normalised 8-point method: centroid in
    double rounded to float32, c = fl32(x - cx), rows (c1x c2x, c1x c2y, c1x, c1y c2x, c1y c2y, c1y, c2x, c2y, 1)."""
    x1 = np.asarray(xy1, dtype=np.float64)
    x2 = np.asarray(xy2, dtype=np.float64)
    c1 = x1.mean(axis=-2).astype(np.float32)
    c2 = x2.mean(axis=-2).astype(np.float32)
    a1 = x1.astype(np.float32) - c1[..., None, :]
    a2 = x2.astype(np.float32) - c2[..., None, :]
    u1, v1, u2, v2 = a1[..., 0], a1[..., 1], a2[..., 0], a2[..., 1]
    A = np.stack([u1 * u2, u1 * v2, u1, v1 * u2, v1 * v2, v1, u2, v2, np.ones_like(u1)], axis=-1).astype(np.float32)

    def T(c):
        t = np.broadcast_to(np.eye(3), c.shape[:-1] + (3, 3)).copy()
        t[..., 0, 2] = -c[..., 0].astype(np.float64)
        t[..., 1, 2] = -c[..., 1].astype(np.float64)
        return t
    return A, T(c1), T(c2)


def estimate(xy1, xy2, return_sv: bool = False):
    """F float32[..., 3, 3] of sampled correspondences [..., P, 2]: null vector of A by numpy's fp64 SVD, largest-magnitude
    component positive (lowest index on ties), F0 = column-major reshape, F = T2^T F0 T1 in fp64 rounded to float32.
    With return_sv also the singular values of A (float64[..., 9], zero-padded when P < 9)."""
    A, T1, T2 = design_matrix(xy1, xy2)
    _, sv, vh = np.linalg.svd(A.astype(np.float64), full_matrices=True)
    v = vh[..., -1, :]
    imax = np.argmax(np.abs(v), axis=-1)
    sign = np.where(np.take_along_axis(v, imax[..., None], axis=-1) < 0, -1.0, 1.0)
    v = v * sign
    F0 = np.swapaxes(v.reshape(v.shape[:-1] + (3, 3)), -1, -2)          # F0[i][j] = v[3 j + i]
    F = (np.swapaxes(T2, -1, -2) @ F0 @ T1).astype(np.float32)
    if not return_sv:
        return F
    pad = np.zeros(sv.shape[:-1] + (9,))
    pad[..., :sv.shape[-1]] = sv
    return F, pad


def rank2(F) -> np.ndarray:
    """Upstream's rank gate on float32 F [..., 3, 3]: #{sigma_k > 3 ulp_f32(sigma_0)} == 2, sigma in fp64."""
    sv = np.linalg.svd(np.asarray(F, dtype=np.float32).astype(np.float64), compute_uv=False)
    tol = (np.spacing(sv[..., 0].astype(np.float32)) * np.float32(3)).astype(np.float64)
    return (sv > tol[..., None]).sum(axis=-1) == 2


def get_fundamental_pairs(all_xy, image_offsets, pair_list, qi, tj, starts, counts, n_samples, pairs_per_sample,
                          threshold, seed, require_rank2=True):
    """Per pair (best, inliers, F float32[3, 3], mask uint8[count], hyp_F float32[S, 3, 3], hyp_counts int32[S]) of
    pgm_ransac_fundamental_pairs_batch_dev, from the oracle's own samples and fp64 estimates."""
    all_xy = np.asarray(all_xy)
    out = []
    for p, (a, b) in enumerate(np.asarray(pair_list).reshape(-1, 2).tolist()):
        st, cnt = int(starts[p]), int(counts[p])
        if cnt < pairs_per_sample:
            out.append((-2, 0, np.zeros((3, 3), np.float32), np.zeros(cnt, np.uint8), None, None))
            continue
        xy1 = all_xy[image_offsets[a] + np.asarray(qi[st:st + cnt], dtype=np.int64)]
        xy2 = all_xy[image_offsets[b] + np.asarray(tj[st:st + cnt], dtype=np.int64)]
        idx = np.stack([sample_indices(cnt, pairs_per_sample, seed, a, b, s) for s in range(n_samples)])
        F = estimate(xy1[idx], xy2[idx])
        valid = rank2(F) if require_rank2 else None
        hc, best, mask = score(F, valid, xy1, xy2, threshold)
        Fb = F[best] if best >= 0 else np.zeros((3, 3), np.float32)
        out.append((best, int(mask.sum()), Fb, mask, F, hc))
    return out


def sign_margin(xy1, xy2) -> np.ndarray:
    """Relative gap between the two largest |v_i| of the null vector of A ([...] per sample).  The sign convention
    (largest-magnitude component positive) is decided by fp64 rounding where it is below ~1e-12: a skew-symmetric F
    (pure translation) has |v_1| == |v_3| and |v_5| == |v_7| up to rounding."""
    A, _, _ = design_matrix(xy1, xy2)
    v = np.abs(np.linalg.svd(A.astype(np.float64), full_matrices=True)[2][..., -1, :])
    top = np.sort(v, axis=-1)
    return (top[..., -1] - top[..., -2]) / top[..., -1]
