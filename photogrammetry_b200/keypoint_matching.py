"""Host mirror of the reference's matcher over the C ABI of libpgmatch.so.

Reference surface (same names, same argument meaning, same error behaviour):

  ImageProcessing.KeypointMatching                       dotnet_src/ImageProcessing/KeypointMatching.cs:8-12
      List<KeypointPair> MatchKeypoints(List<Keypoint>, List<Keypoint>)        :14-69
  photogrammetry.image_processing.keypoint_matching.match_keypoints            python_src/.../keypoint_matching.py:7-33

``KeypointMatching().MatchKeypoints(kp1, kp2)`` returns exactly ``len(kp1)``
``KeypointPair`` objects whose ``Keypoint1``/``Keypoint2`` are *the caller's own
objects* (KeypointMatching.cs:57-62), in the reference's order, including the
``(keypoints1[0], keypoints2[0], int.MaxValue)`` tail when ``len(kp1) > len(kp2)``
and an ``IndexError`` (the reference: ArgumentOutOfRangeException, :61) when
``kp2`` is empty and ``kp1`` is not.

All compute happens in CUDA kernels behind ``pgm_*``; nothing here touches
``oracle/`` and there is no CPU path.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import (PGM_E_CAPACITY, PGM_E_EMPTY_TRAIN, PGM_FLAG_PYTHON_GENERATION, PGM_FLAG_REFERENCE_COMPAT_TAIL,
                   PGM_OK, EmptyTrainError, PgmatchError, PgmatchLibraryError, Stats)
from .descriptors import as_descriptor_rows, pack_descriptors
from .keypoint import Keypoint, KeypointPair


def _addr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


class Matcher:
    """One ``pgm_handle``: a device, a stream and its scratch memory (not thread-affine)."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        rc = self._lib.pgm_create(int(device), C.byref(self._h))
        if rc != PGM_OK:
            self._h = C.c_void_p()
            raise PgmatchLibraryError(
                f"pgm_create(device={device}) failed: {self._lib.pgm_status_string(rc).decode()} "
                "(libpgmatch has no CPU fallback)")
        self.device = int(device)
        self._user_stream: Optional[int] = None     # what set_stream() bound (None: the handle's own stream)

    # -- lifetime ---------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.pgm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- helpers ----------------------------------------------------------
    def _check(self, rc: int) -> None:
        if rc == PGM_OK:
            return
        msg = self._lib.pgm_last_error(self._h).decode() or self._lib.pgm_status_string(rc).decode()
        if rc == PGM_E_EMPTY_TRAIN:
            raise EmptyTrainError(rc, msg)
        raise PgmatchError(rc, msg)

    def set_stream(self, cuda_stream: Optional[int]) -> None:
        """Run on a caller-owned CUDA stream (e.g. ``torch.cuda.Stream().cuda_stream``).  ``None`` returns to the
        handle's own stream; ``0`` (what torch reports for its default stream) selects the legacy default
        stream explicitly (``cudaStreamLegacy``), because a NULL stream means "own stream" across the ABI."""
        if cuda_stream is None:
            addr = 0
        elif int(cuda_stream) == 0:
            addr = 1                    # cudaStreamLegacy
        else:
            addr = int(cuda_stream)
        self._check(self._lib.pgm_set_stream(self._h, C.c_void_p(addr)))
        self._user_stream = None if cuda_stream is None else int(cuda_stream)

    @contextlib.contextmanager
    def torch_ordered(self, device=None):
        """Entry points that take or return torch tensors must be ordered against torch's work.  If the caller
        bound a stream with :meth:`set_stream` that is their contract; otherwise the handle is bound to torch's
        CURRENT stream for the duration of the call, so inputs written by torch kernels are visible and the
        returned tensors can be consumed by torch (or NCCL) without an extra synchronisation."""
        if self._user_stream is not None:
            yield
            return
        import torch
        cur = torch.cuda.current_stream(torch.device("cuda", self.device) if device is None else device).cuda_stream
        self._check(self._lib.pgm_set_stream(self._h, C.c_void_p(1 if int(cur) == 0 else int(cur))))
        try:
            yield
        finally:
            self._check(self._lib.pgm_set_stream(self._h, C.c_void_p(0)))

    def synchronize(self) -> None:
        self._check(self._lib.pgm_synchronize(self._h))

    def stats(self) -> dict:
        st = Stats()
        self._check(self._lib.pgm_get_stats(self._h, C.byref(st)))
        return st.as_dict()

    # -- MatchKeypoints on packed rows ------------------------------------
    def match_greedy(self, q: np.ndarray, t: np.ndarray, desc_bits: Optional[int] = None,
                     reference_compat_tail: bool = True, out: Optional[np.ndarray] = None) -> np.ndarray:
        """``int32[count, 3]`` rows (query index, train index, distance) in the reference's order.

        ``out``: optional caller-owned C-contiguous ``int32[3, >= n1]`` array (e.g. from
        :func:`photogrammetry_b200._lib.pinned_empty`); the call then returns the SoA view ``out[:, :count]``
        with no further copy.  Page-locked inputs and outputs are transferred without staging."""
        q, bits_q = as_descriptor_rows(q, desc_bits)
        t, bits_t = as_descriptor_rows(t, desc_bits)
        n1, n2 = int(q.shape[0]), int(t.shape[0])
        stride = int(q.shape[1]) if n1 else int(t.shape[1])
        if n1 and n2 and q.shape[1] != t.shape[1]:
            raise ValueError("query and train descriptors have different strides")
        bits = desc_bits or max(bits_q, bits_t)
        reuse = out is not None
        if reuse:
            if out.dtype != np.int32 or out.ndim != 2 or out.shape[0] != 3 or out.shape[1] < n1 or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous int32[3, >= n1] array")
        else:
            out = np.empty((3, max(n1, 1)), dtype=np.int32)
        cnt = C.c_int32(0)
        flags = PGM_FLAG_REFERENCE_COMPAT_TAIL if reference_compat_tail else 0
        self._check(self._lib.pgm_match_hamming_greedy(
            self._h, _addr(q), n1, _addr(t), n2, bits, stride,
            out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data, n1, C.byref(cnt), flags))
        if reuse:
            return out[:, :cnt.value]
        return np.ascontiguousarray(out[:, :cnt.value].T)

    def match_greedy_dev(self, d_q: int, n1: int, d_t: int, n2: int, desc_bits: int, stride: int,
                         d_out_qi: int, d_out_tj: int, d_out_dist: int, capacity: int,
                         reference_compat_tail: bool = True) -> int:
        """Device-pointer variant (raw addresses).  Returns the number of triples written."""
        cnt = C.c_int32(0)
        flags = PGM_FLAG_REFERENCE_COMPAT_TAIL if reference_compat_tail else 0
        self._check(self._lib.pgm_match_hamming_greedy_dev(
            self._h, d_q, n1, d_t, n2, desc_bits, stride, d_out_qi, d_out_tj, d_out_dist, capacity,
            C.byref(cnt), flags))
        return cnt.value

    def match_pairs_batch(self, all_desc: np.ndarray, image_offsets: Sequence[int], pair_list,
                          desc_bits: Optional[int] = None, reference_compat_tail: bool = True,
                          out: Optional[np.ndarray] = None):
        """Match many image pairs in one call.

        Returns ``(triples int32[total, 3], starts int64[n_pairs], counts int32[n_pairs])``;
        pair ``p`` owns ``triples[starts[p]:starts[p]+counts[p]]``.

        ``out``: optional caller-owned ``int32[3, >= total]`` C-contiguous array that receives the raw SoA
        output (qi, tj, dist) and is reused across calls; the function then returns ``out[:, :total]`` itself
        (SoA, no copy) in place of the ``[total, 3]`` array.  Gigabyte-sized result arrays are dominated by
        the operating system's first-touch page faults when they are allocated fresh on every call.
        """
        all_desc, bits = as_descriptor_rows(all_desc, desc_bits)
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        pairs = np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
        n_images, n_pairs = len(offs) - 1, len(pairs)
        sizes = np.diff(offs)
        n1s = sizes[pairs[:, 0]] if n_pairs else np.zeros(0, dtype=np.int64)
        starts = np.concatenate([[0], np.cumsum(n1s)]).astype(np.int64)
        total = int(starts[-1])
        reuse = out is not None
        if reuse:
            if out.dtype != np.int32 or out.ndim != 2 or out.shape[0] != 3 or out.shape[1] < total or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous int32[3, >= total] array")
        else:
            out = np.empty((3, max(total, 1)), dtype=np.int32)
        counts = np.zeros(max(n_pairs, 1), dtype=np.int32)
        flags = PGM_FLAG_REFERENCE_COMPAT_TAIL if reference_compat_tail else 0
        self._check(self._lib.pgm_match_pairs_batch(
            self._h, _addr(all_desc), offs.ctypes.data, n_images, pairs.ctypes.data, n_pairs,
            desc_bits or bits, int(all_desc.shape[1]), out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data,
            total, counts.ctypes.data, flags))
        if reuse:
            return out[:, :total], starts[:-1], counts[:n_pairs]
        return np.ascontiguousarray(out[:, :total].T), starts[:-1], counts[:n_pairs]

    def match_pairs_batch_dev(self, d_all_desc: int, image_offsets, pair_list, desc_bits: int, stride: int,
                              d_out_qi: int, d_out_tj: int, d_out_dist: int, capacity: int,
                              reference_compat_tail: bool = True) -> np.ndarray:
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        pairs = np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
        counts = np.zeros(max(len(pairs), 1), dtype=np.int32)
        flags = PGM_FLAG_REFERENCE_COMPAT_TAIL if reference_compat_tail else 0
        self._check(self._lib.pgm_match_pairs_batch_dev(
            self._h, d_all_desc, offs.ctypes.data, len(offs) - 1, pairs.ctypes.data, len(pairs), desc_bits, stride,
            d_out_qi, d_out_tj, d_out_dist, capacity, counts.ctypes.data, flags))
        return counts[:len(pairs)]

    # -- nearest / second nearest, ratio, cross-check ----------------------
    def knn2(self, q: np.ndarray, t: np.ndarray, desc_bits: Optional[int] = None):
        q, bits_q = as_descriptor_rows(q, desc_bits)
        t, bits_t = as_descriptor_rows(t, desc_bits)
        n1, n2 = int(q.shape[0]), int(t.shape[0])
        stride = int(q.shape[1]) if n1 else int(t.shape[1])
        out = np.empty((4, max(n1, 1)), dtype=np.int32)
        self._check(self._lib.pgm_knn2_hamming(self._h, _addr(q), n1, _addr(t), n2, desc_bits or max(bits_q, bits_t),
                                               stride, *(out[k].ctypes.data for k in range(4))))
        return tuple(out[k, :n1].copy() for k in range(4))

    def match_ratio_crosscheck(self, q: np.ndarray, t: np.ndarray, ratio: float = 0.8, cross_check: bool = True,
                               max_dist: int = -1, desc_bits: Optional[int] = None) -> np.ndarray:
        q, bits_q = as_descriptor_rows(q, desc_bits)
        t, bits_t = as_descriptor_rows(t, desc_bits)
        n1, n2 = int(q.shape[0]), int(t.shape[0])
        stride = int(q.shape[1]) if n1 else int(t.shape[1])
        out = np.empty((3, max(n1, 1)), dtype=np.int32)
        cnt = C.c_int32(0)
        self._check(self._lib.pgm_match_ratio_crosscheck(
            self._h, _addr(q), n1, _addr(t), n2, desc_bits or max(bits_q, bits_t), stride, float(ratio),
            int(bool(cross_check)), int(max_dist), out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data,
            n1, C.byref(cnt)))
        return np.ascontiguousarray(out[:, :cnt.value].T)

    # -- device-resident forms (torch tensors on this matcher's GPU; used by sharding.TrainShardedKnn) --
    def knn2_hamming_dev(self, d_q, d_t, desc_bits: int = 256):
        """(best_j, best_d, second_j, second_d) as int32 tensors; ``d_q``/``d_t``: uint8 ``[n, stride]`` on the GPU."""
        import torch
        n1, n2 = int(d_q.shape[0]), int(d_t.shape[0])
        stride = int(d_q.shape[1]) if n1 else int(d_t.shape[1])
        out = torch.empty((4, max(n1, 1)), dtype=torch.int32, device=d_q.device)
        with self.torch_ordered(d_q.device):
            self._check(self._lib.pgm_knn2_hamming_dev(self._h, d_q.data_ptr() if n1 else None, n1,
                                                       d_t.data_ptr() if n2 else None, n2, int(desc_bits), stride,
                                                       *(out[k].data_ptr() for k in range(4))))
        return tuple(out[k, :n1] for k in range(4))

    def pack_top2_keys_dev(self, best_j, best_d, second_j, second_d, index_offset: int):
        """int32 ``[2, n]`` exchange keys (distance << 20 | global train index, 0x7F7F7F7F = absent)."""
        import torch
        n = int(best_j.shape[0])
        keys = torch.empty((2, max(n, 1)), dtype=torch.int32, device=best_j.device)
        with self.torch_ordered(best_j.device):
            self._check(self._lib.pgm_pack_top2_keys_dev(self._h, best_j.data_ptr(), best_d.data_ptr(),
                                                         second_j.data_ptr(), second_d.data_ptr(), n, int(index_offset),
                                                         keys.data_ptr()))
        return keys[:, :n] if n else keys[:, :0]

    def merge_top2_dev(self, keys):
        """``keys``: int32 ``[n_shards, 2, n]`` (contiguous) -> the merged (best_j, best_d, second_j, second_d)."""
        import torch
        g, _, n = (int(x) for x in keys.shape)
        keys = keys.contiguous()
        out = torch.empty((4, max(n, 1)), dtype=torch.int32, device=keys.device)
        with self.torch_ordered(keys.device):
            self._check(self._lib.pgm_merge_top2_dev(self._h, keys.data_ptr(), g, n, *(out[k].data_ptr() for k in range(4))))
        return tuple(out[k, :n] for k in range(4))

    def ratio_crosscheck_filter_dev(self, n2: int, best_j, best_d, second_d, col_best_i, ratio: float = 0.8,
                                    cross_check: bool = True, max_dist: int = -1):
        """The filter of ``match_ratio_crosscheck`` on device-resident knn2 results -> int32 ``[3, count]``."""
        import torch
        n1 = int(best_j.shape[0])
        out = torch.empty((3, max(n1, 1)), dtype=torch.int32, device=best_j.device)
        cnt = C.c_int32(0)
        with self.torch_ordered(best_j.device):
            self._check(self._lib.pgm_ratio_crosscheck_filter_dev(
                self._h, n1, int(n2), best_j.data_ptr(), best_d.data_ptr(), second_d.data_ptr(),
                col_best_i.data_ptr() if col_best_i is not None and col_best_i.numel() else None, float(ratio),
                int(bool(cross_check)), int(max_dist), out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                C.byref(cnt)))
        return out[:, :cnt.value]

    def match_ratio_crosscheck_batch_dev(self, d_all_desc, image_offsets, pair_list, desc_bits: int = 256, ratio: float = 0.8,
                                         cross_check: bool = True, max_dist: int = -1):
        """Nearest neighbour + ratio test + cross-check for many small pairs in ONE launch (a frame sequence).
        ``d_all_desc``: torch uint8 ``[sum, stride]`` on the GPU.  Returns ``(out int32[3, sum of n1], starts int64[n_pairs],
        counts int32[n_pairs])``; pair ``p`` owns ``out[:, starts[p]:starts[p] + counts[p]]`` (ascending query index)."""
        return self._ratio_batch_dev(self._lib.pgm_match_ratio_crosscheck_batch_dev, d_all_desc, image_offsets, pair_list,
                                     desc_bits, ratio, cross_check, max_dist)

    def match_ratio_crosscheck_pairs_batch_dev(self, d_all_desc, image_offsets, pair_list, desc_bits: int = 256,
                                               ratio: float = 0.8, cross_check: bool = True, max_dist: int = -1):
        """:meth:`match_ratio_crosscheck_batch_dev` for pairs of any size (e.g. all pairs of a large image set): one
        fused distance pass per chunk of pairs instead of one CTA per pair.  Same arguments, same return value; per pair
        the same triples as :meth:`match_ratio_crosscheck`."""
        return self._ratio_batch_dev(self._lib.pgm_match_ratio_crosscheck_pairs_batch_dev, d_all_desc, image_offsets,
                                     pair_list, desc_bits, ratio, cross_check, max_dist)

    def _ratio_batch_dev(self, fn, d_all_desc, image_offsets, pair_list, desc_bits, ratio, cross_check, max_dist):
        import torch
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        pairs = np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
        sizes = np.diff(offs)
        n1s = sizes[pairs[:, 0]] if len(pairs) else np.zeros(0, np.int64)
        starts = np.concatenate([[0], np.cumsum(n1s)]).astype(np.int64)
        total = int(starts[-1])
        out = torch.empty((3, max(total, 1)), dtype=torch.int32, device=d_all_desc.device)
        counts = np.zeros(max(len(pairs), 1), dtype=np.int32)
        with self.torch_ordered(d_all_desc.device):
            self._check(fn(
                self._h, d_all_desc.data_ptr(), offs.ctypes.data, len(offs) - 1, pairs.ctypes.data, len(pairs), int(desc_bits),
                int(d_all_desc.shape[1]), float(ratio), int(bool(cross_check)), int(max_dist), out[0].data_ptr(),
                out[1].data_ptr(), out[2].data_ptr(), total, counts.ctypes.data))
        return out, starts[:-1], counts[:len(pairs)]

    def match_keypoints_sorted(self, q: np.ndarray, t: np.ndarray, desc_bits: Optional[int] = None) -> np.ndarray:
        """``int64[n1, n2, 2]`` = (idx2, dist), rows sorted by (dist, idx2) (keypoint_matching.py:7-33)."""
        q, bits_q = as_descriptor_rows(q, desc_bits)
        t, bits_t = as_descriptor_rows(t, desc_bits)
        n1, n2 = int(q.shape[0]), int(t.shape[0])
        stride = int(q.shape[1]) if n1 else int(t.shape[1])
        out = np.zeros((n1, n2, 2), dtype=np.int64)
        self._check(self._lib.pgm_match_keypoints_sorted(self._h, _addr(q), n1, _addr(t), n2,
                                                         desc_bits or max(bits_q, bits_t), stride, out.ctypes.data))
        return out

    def knn2_l2(self, q: np.ndarray, t: np.ndarray):
        """Float descriptors: (best_j, best_d, second_j, second_d) under squared L2 (tcgen05 GEMM + exact refinement)."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        t = np.ascontiguousarray(t, dtype=np.float32)
        n1, n2 = int(q.shape[0]), int(t.shape[0])
        dim = int(q.shape[1]) if n1 else int(t.shape[1])
        bj = np.empty(max(n1, 1), dtype=np.int32); sj = np.empty(max(n1, 1), dtype=np.int32)
        bd = np.empty(max(n1, 1), dtype=np.float32); sd = np.empty(max(n1, 1), dtype=np.float32)
        self._check(self._lib.pgm_knn2_l2(self._h, _addr(q), n1, _addr(t), n2, dim, bj.ctypes.data, bd.ctypes.data,
                                          sj.ctypes.data, sd.ctypes.data))
        return bj[:n1], bd[:n1], sj[:n1], sd[:n1]

    def knn2_l2_pairs_batch_dev(self, d_all_desc, image_offsets, pair_list):
        """:meth:`knn2_l2` for many image pairs in one call.  ``d_all_desc``: torch float32 ``[rows, dim]`` on the GPU
        (``dim <= 128``), image ``k`` = rows ``image_offsets[k]:image_offsets[k + 1]``.  Returns ``(best_j, best_d,
        second_j, second_d, starts)``: tensors of ``sum of n1`` rows; pair ``p``'s query rows start at ``starts[p]``.
        Per pair the result is bit-identical to :meth:`knn2_l2` on the CTA-pair path (``n1 > 128``)."""
        import torch
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        pairs = np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
        starts = self._pair_starts(offs, pairs)
        total = int(starts[-1])
        dev = d_all_desc.device
        bj = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        sj = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        bd = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
        sd = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
        with self.torch_ordered(dev):
            self._check(self._lib.pgm_knn2_l2_pairs_batch_dev(
                self._h, d_all_desc.data_ptr(), offs.ctypes.data, len(offs) - 1, pairs.ctypes.data, len(pairs),
                int(d_all_desc.shape[1]), bj.data_ptr(), bd.data_ptr(), sj.data_ptr(), sd.data_ptr(), total))
        return bj[:total], bd[:total], sj[:total], sd[:total], starts[:-1]

    def match_l2_ratio_crosscheck_pairs_batch_dev(self, d_all_desc, image_offsets, pair_list, ratio: float = 0.8,
                                                  cross_check: bool = True, max_sq_dist: float = -1.0):
        """Float descriptors: nearest neighbour + Lowe's ratio test + cross-check for many image pairs in one call.
        ``d_all_desc`` as in :meth:`knn2_l2_pairs_batch_dev`.  Keeps ``(i, j1, d1)`` iff ``n2 < 2 or ratio <= 0 or
        d1 < ratio^2 d2`` (squared distances, fp32), ``j1``'s nearest query is ``i`` (with ``cross_check``) and
        ``max_sq_dist < 0 or d1 <= max_sq_dist``.  Returns ``(qi int32, tj int32, dist float32, starts int64[n_pairs],
        counts int32[n_pairs])``; pair ``p`` owns ``[starts[p], starts[p] + counts[p])`` in ascending ``qi``."""
        import torch
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        pairs = np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
        starts = self._pair_starts(offs, pairs)
        total = int(starts[-1])
        dev = d_all_desc.device
        qi = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        tj = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        dist = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
        counts = np.zeros(max(len(pairs), 1), dtype=np.int32)
        with self.torch_ordered(dev):
            self._check(self._lib.pgm_match_l2_ratio_crosscheck_pairs_batch_dev(
                self._h, d_all_desc.data_ptr(), offs.ctypes.data, len(offs) - 1, pairs.ctypes.data, len(pairs),
                int(d_all_desc.shape[1]), float(ratio), int(bool(cross_check)), float(max_sq_dist), qi.data_ptr(),
                tj.data_ptr(), dist.data_ptr(), total, counts.ctypes.data))
        return qi, tj, dist, starts[:-1], counts[:len(pairs)]

    @staticmethod
    def _pair_starts(offs, pairs):
        sizes = np.diff(offs)
        n1s = sizes[pairs[:, 0]] if len(pairs) else np.zeros(0, np.int64)
        return np.concatenate([[0], np.cumsum(n1s)]).astype(np.int64)

    def l2_last_fallback_rows(self) -> int:
        """Queries of the last float call that were recomputed exhaustively (their candidate band could not be
        certified from the kernel's top-8 lists; a batch call counts all its chunks and both directions); -1 if that
        call used the three-term bf16 ranking."""
        return int(self._lib.pgm_l2_last_fallback_rows(self._h))

    # -- the producer of the matcher's inputs: FAST-12, BRIEF, NMS ----------
    def fast_detect(self, gray: np.ndarray, threshold: float, python_generation: bool = False):
        """``KeypointDetection.Detect`` without the descriptors (KeypointDetection.cs:42-133).
        gray: ``float32[H, W]``.  Returns (xy int32[n, 2] as (x, y) in row-major scan order, score int32[n])."""
        gray = np.ascontiguousarray(gray, dtype=np.float32)
        if gray.ndim != 2:
            raise ValueError("gray must be a 2-D array [height, width]")
        hgt, wid = gray.shape
        flags = PGM_FLAG_PYTHON_GENERATION if python_generation else 0
        cap = 4096
        while True:
            xy = np.empty((cap, 2), dtype=np.int32)
            sc = np.empty(cap, dtype=np.int32)
            cnt = C.c_int32(0)
            rc = self._lib.pgm_fast_detect(self._h, gray.ctypes.data, wid, hgt, float(threshold), flags,
                                           xy.ctypes.data, sc.ctypes.data, cap, C.byref(cnt))
            if rc == PGM_E_CAPACITY and cnt.value > cap:
                cap = cnt.value
                continue
            self._check(rc)
            return xy[:cnt.value].copy(), sc[:cnt.value].copy()

    def brief_describe(self, gray: np.ndarray, xy: np.ndarray, pairs: np.ndarray, stride: Optional[int] = None,
                       python_generation: bool = False) -> np.ndarray:
        """``Keypoint.GetBriefDescriptor`` (Keypoint.cs:29-57) for every (x, y) of ``xy``.
        pairs: int32[n_pairs, 4] = (dx1, dy1, dx2, dy2).  Returns ``uint8[n, stride]`` matcher rows."""
        gray = np.ascontiguousarray(gray, dtype=np.float32)
        xy = np.ascontiguousarray(xy, dtype=np.int32).reshape(-1, 2)
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 4)
        hgt, wid = gray.shape
        n, n_pairs = len(xy), len(pairs)
        stride = stride or ((n_pairs + 127) // 128) * 16
        out = np.zeros((n, stride), dtype=np.uint8)
        flags = PGM_FLAG_PYTHON_GENERATION if python_generation else 0
        self._check(self._lib.pgm_brief_describe(self._h, gray.ctypes.data, wid, hgt, _addr(xy), n, pairs.ctypes.data,
                                                 n_pairs, stride, flags, _addr(out)))
        return out

    def detect_describe_dev(self, d_gray, threshold: float, pairs: np.ndarray, nms_radius: int = -1,
                            stride: Optional[int] = None, python_generation: bool = False, capacity: int = 8192):
        """FAST-12 -> (NMS when ``nms_radius >= 0``) -> BRIEF on a device-resident image (torch float32 ``[H, W]``
        on this matcher's GPU).  Returns torch tensors ``(xy int32[n, 2], score int32[n], desc uint8[n, stride])``
        on the device, in the reference's output order; ``desc`` is directly a matcher operand."""
        import torch
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 4)
        hgt, wid = (int(x) for x in d_gray.shape)
        n_pairs = len(pairs)
        stride = stride or ((n_pairs + 127) // 128) * 16
        flags = PGM_FLAG_PYTHON_GENERATION if python_generation else 0
        d_gray = d_gray.contiguous()
        cap = int(capacity)
        while True:
            xy = torch.empty((max(cap, 1), 2), dtype=torch.int32, device=d_gray.device)
            sc = torch.empty(max(cap, 1), dtype=torch.int32, device=d_gray.device)
            desc = torch.zeros((max(cap, 1), stride), dtype=torch.uint8, device=d_gray.device)
            cnt = C.c_int32(0)
            with self.torch_ordered(d_gray.device):
                rc = self._lib.pgm_detect_describe_dev(self._h, d_gray.data_ptr(), wid, hgt, float(threshold),
                                                       int(nms_radius), pairs.ctypes.data, n_pairs, stride, flags,
                                                       xy.data_ptr(), sc.data_ptr(), desc.data_ptr(), cap, C.byref(cnt))
            if rc == PGM_E_CAPACITY and cnt.value > cap:
                cap = cnt.value
                continue
            self._check(rc)
            n = cnt.value
            return xy[:n], sc[:n], desc[:n]

    def detect_describe_batch_dev(self, d_gray, threshold: float, pairs: np.ndarray, capacity: int = 4096,
                                  stride: Optional[int] = None, python_generation: bool = False, read_counts: bool = True,
                                  nms_radius: int = -1):
        """FAST-12 -> BRIEF for a stack of device-resident images (torch float32 ``[K, H, W]``), one call, nothing read
        back between the images.  Returns ``(xy int32[K, capacity, 2], score int32[K, capacity], desc uint8[K, capacity,
        stride], counts)`` where ``counts`` is a numpy int32[K] (one synchronisation) or, with ``read_counts=False``,
        a device tensor (no synchronisation at all).  A count above ``capacity`` means that image's list was truncated.

        With ``nms_radius >= 0`` the chain includes the reference's NMS (RedundantKeypointEliminator) on every image's
        full FAST list, as :meth:`detect_describe_dev` does per image: the counts are then the survivors, in the
        reference's output order, and the call synchronises once more, to size its scratch from the FAST totals."""
        import torch
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 4)
        k, hgt, wid = (int(x) for x in d_gray.shape)
        n_pairs = len(pairs)
        stride = stride or ((n_pairs + 127) // 128) * 16
        flags = PGM_FLAG_PYTHON_GENERATION if python_generation else 0
        d_gray = d_gray.contiguous()
        cap = max(int(capacity), 1)
        xy = torch.empty((k, cap, 2), dtype=torch.int32, device=d_gray.device)
        sc = torch.empty((k, cap), dtype=torch.int32, device=d_gray.device)
        desc = torch.zeros((k, cap, stride), dtype=torch.uint8, device=d_gray.device)
        d_cnt = torch.zeros(max(k, 1), dtype=torch.int32, device=d_gray.device)
        h_cnt = np.zeros(max(k, 1), dtype=np.int32)
        with self.torch_ordered(d_gray.device):
            if nms_radius >= 0:
                rc = self._lib.pgm_detect_nms_describe_batch_dev(
                    self._h, d_gray.data_ptr(), k, wid, hgt, float(threshold), int(nms_radius), pairs.ctypes.data, n_pairs,
                    stride, flags, xy.data_ptr(), sc.data_ptr(), desc.data_ptr(), cap, d_cnt.data_ptr(),
                    h_cnt.ctypes.data if read_counts else None)
            else:
                rc = self._lib.pgm_detect_describe_batch_dev(
                    self._h, d_gray.data_ptr(), k, wid, hgt, float(threshold), pairs.ctypes.data, n_pairs, stride, flags,
                    xy.data_ptr(), sc.data_ptr(), desc.data_ptr(), cap, d_cnt.data_ptr(),
                    h_cnt.ctypes.data if read_counts else None)
            self._check(rc)
        return xy, sc, desc, (h_cnt[:k] if read_counts else d_cnt[:k])

    def detect_describe_images_batch_dev(self, images, threshold: float, pairs: np.ndarray, capacity: int = 4096,
                                         stride: Optional[int] = None, python_generation: bool = False,
                                         read_counts: bool = True, nms_radius: int = -1):
        """:meth:`detect_describe_batch_dev` for images of any sizes: ``images`` is a list of 2-D torch float32 tensors on
        this matcher's GPU, each detected at its own size (portrait next to landscape, mixed cameras and crops), in one
        call.  They are packed into one flat device buffer.  Arguments, return value and synchronisation are those of
        :meth:`detect_describe_batch_dev`; per image the result equals :meth:`detect_describe_dev` on that image."""
        import torch
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 4)
        k = len(images)
        if any(im.dim() != 2 or im.dtype != torch.float32 for im in images):
            raise ValueError("images must be 2-D float32 tensors")
        heights = np.array([int(im.shape[0]) for im in images], dtype=np.int32)
        widths = np.array([int(im.shape[1]) for im in images], dtype=np.int32)
        offs = np.zeros(k + 1, dtype=np.int64)
        offs[1:] = np.cumsum(widths.astype(np.int64) * heights)
        n_pairs = len(pairs)
        stride = stride or ((n_pairs + 127) // 128) * 16
        flags = PGM_FLAG_PYTHON_GENERATION if python_generation else 0
        dev = images[0].device if k else torch.device("cuda", self.device)
        cap = max(int(capacity), 1)
        with self.torch_ordered(dev):
            d_gray = torch.cat([im.reshape(-1) for im in images]) if k else torch.empty(1, dtype=torch.float32, device=dev)
            xy = torch.empty((k, cap, 2), dtype=torch.int32, device=dev)
            sc = torch.empty((k, cap), dtype=torch.int32, device=dev)
            desc = torch.zeros((k, cap, stride), dtype=torch.uint8, device=dev)
            d_cnt = torch.zeros(max(k, 1), dtype=torch.int32, device=dev)
            h_cnt = np.zeros(max(k, 1), dtype=np.int32)
            self._check(self._lib.pgm_detect_describe_images_batch_dev(
                self._h, d_gray.data_ptr(), offs.ctypes.data, widths.ctypes.data, heights.ctypes.data, k, float(threshold),
                int(nms_radius), pairs.ctypes.data, n_pairs, stride, flags, xy.data_ptr(), sc.data_ptr(), desc.data_ptr(),
                cap, d_cnt.data_ptr(), h_cnt.ctypes.data if read_counts else None))
        return xy, sc, desc, (h_cnt[:k] if read_counts else d_cnt[:k])

    def nms(self, xy: np.ndarray, score: np.ndarray, radius: int) -> np.ndarray:
        """``RedundantKeypointEliminator.EliminateRedundantKeypoints`` (RedundantKeypointEliminator.cs:16-39):
        indices of the surviving keypoints in the reference's output order."""
        xy = np.ascontiguousarray(xy, dtype=np.int32).reshape(-1, 2)
        score = np.ascontiguousarray(score, dtype=np.int32).reshape(-1)
        n = len(xy)
        if len(score) != n:
            raise ValueError("xy and score differ in length")
        kept = np.empty(max(n, 1), dtype=np.int32)
        cnt = C.c_int32(0)
        self._check(self._lib.pgm_nms(self._h, _addr(xy), _addr(score), n, int(radius), kept.ctypes.data,
                                      C.byref(cnt)))
        return kept[:cnt.value].copy()

    # -- the consumer of the match list: RANSAC hypothesis scoring -----------
    def ransac_score(self, F: np.ndarray, xy1: np.ndarray, xy2: np.ndarray, threshold: float,
                     valid: Optional[np.ndarray] = None):
        """Scoring loops of ``CameraPoseEstimation.GetFundamentalMatrix`` (CameraPoseEstimation.cs:41-88).
        Returns (counts int32[n_hyp], best index or -1, inlier mask uint8[n] of the best hypothesis)."""
        F = np.ascontiguousarray(F, dtype=np.float32).reshape(-1, 9)
        xy1 = np.ascontiguousarray(xy1, dtype=np.int32).reshape(-1, 2)
        xy2 = np.ascontiguousarray(xy2, dtype=np.int32).reshape(-1, 2)
        if len(xy1) != len(xy2):
            raise ValueError("xy1 and xy2 differ in length")
        v = None if valid is None else np.ascontiguousarray(valid, dtype=np.uint8).reshape(-1)
        if v is not None and len(v) != len(F):
            raise ValueError("valid and F differ in length")
        counts = np.empty(max(len(F), 1), dtype=np.int32)
        mask = np.zeros(max(len(xy1), 1), dtype=np.uint8)
        best = C.c_int32(-1)
        self._check(self._lib.pgm_ransac_score(self._h, _addr(F), _addr(v), len(F), _addr(xy1), _addr(xy2), len(xy1),
                                               float(threshold), counts.ctypes.data, C.byref(best), mask.ctypes.data))
        return counts[:len(F)], int(best.value), mask[:len(xy1)]

    def ransac_fundamental_pairs_batch_dev(self, d_xy, image_offsets, pair_list, qi, tj, starts, counts,
                                           n_samples: int = 2000, pairs_per_sample: int = 32, threshold: float = 0.001,
                                           seed: int = 0, require_rank2: bool = True, hypotheses: bool = False):
        """``GetFundamentalMatrix(list, n_samples, pairs_per_sample, threshold)`` (CameraPoseEstimation.cs:26-94) for
        many match lists in one call, on the device and with no read-back.  The defaults are upstream's call
        (Program.cs: 2000, 32, 0.001f) and the host mirror's rank gate.

        ``d_xy``: torch int32 ``[rows, 2]`` keypoint coordinates, image ``k`` at rows ``image_offsets[k]:image_offsets[k+1]``;
        ``qi``/``tj``: torch int32 match indices (e.g. rows 0 and 1 of what the batch matchers return) with ``starts`` /
        ``counts`` as those methods return them.  Returns torch tensors ``(best int32[n_pairs], inliers int32[n_pairs],
        F float32[n_pairs, 3, 3], mask uint8[capacity])`` -- ``best`` is the winning sample, -1 if no sample has an inlier,
        -2 if the pair has fewer than ``pairs_per_sample`` matches -- plus ``(hyp_F float32[n_pairs, S, 3, 3],
        hyp_counts int32[n_pairs, S])`` with ``hypotheses=True`` (rows of pairs below ``pairs_per_sample`` stay zero)."""
        import torch
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        pairs = np.ascontiguousarray(pair_list, dtype=np.int32).reshape(-1, 2)
        st = np.ascontiguousarray(starts, dtype=np.int64).reshape(-1)
        cn = np.ascontiguousarray(counts, dtype=np.int32).reshape(-1)
        n_pairs = len(pairs)
        if len(st) != n_pairs or len(cn) != n_pairs:
            raise ValueError("starts and counts need one entry per pair")
        for name, t in (("d_xy", d_xy), ("qi", qi), ("tj", tj)):
            if t.dtype != torch.int32 or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous int32 tensor")
        capacity = min(int(qi.numel()), int(tj.numel()))
        dev = d_xy.device
        S = int(n_samples)
        best = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=dev)
        inliers = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=dev)
        F = torch.empty((max(n_pairs, 1), 3, 3), dtype=torch.float32, device=dev)
        mask = torch.zeros(max(capacity, 1), dtype=torch.uint8, device=dev)
        hyp_F = hyp_c = None
        if hypotheses:
            hyp_F = torch.zeros((max(n_pairs, 1), max(S, 1), 3, 3), dtype=torch.float32, device=dev)
            hyp_c = torch.zeros((max(n_pairs, 1), max(S, 1)), dtype=torch.int32, device=dev)
        flags = _lib.PGM_FLAG_RANSAC_RANK_TEST if require_rank2 else 0
        with self.torch_ordered(dev):
            self._check(self._lib.pgm_ransac_fundamental_pairs_batch_dev(
                self._h, d_xy.data_ptr(), offs.ctypes.data, len(offs) - 1, pairs.ctypes.data, n_pairs, qi.data_ptr(),
                tj.data_ptr(), st.ctypes.data, cn.ctypes.data, S, int(pairs_per_sample), float(threshold),
                int(seed) & 0xFFFFFFFFFFFFFFFF, flags, best.data_ptr(), inliers.data_ptr(), F.data_ptr(), mask.data_ptr(),
                capacity, hyp_F.data_ptr() if hypotheses else None, hyp_c.data_ptr() if hypotheses else None))
        out = (best[:n_pairs], inliers[:n_pairs], F[:n_pairs], mask[:capacity])
        if hypotheses:
            out += (hyp_F[:n_pairs], hyp_c[:n_pairs])
        return out

    def set_profiling(self, enabled: bool) -> None:
        self._check(self._lib.pgm_set_profiling(self._h, int(bool(enabled))))

    def round_profile(self):
        """(ms float32[k], evals int64[k]) per round-kernel launch of the last greedy call."""
        ms = np.zeros(256, dtype=np.float32)
        ev = np.zeros(256, dtype=np.int64)
        n = C.c_int32(0)
        self._check(self._lib.pgm_get_round_profile(self._h, ms.ctypes.data, ev.ctypes.data, 256, C.byref(n)))
        return ms[:n.value].copy(), ev[:n.value].copy()

    def measure_popc_peak(self, millis: int = 200):
        p, l = C.c_double(0), C.c_double(0)
        self._check(self._lib.pgm_measure_popc_peak(self._h, int(millis), C.byref(p), C.byref(l)))
        return p.value, l.value


_default: dict = {}


def default_matcher(device: int = 0) -> Matcher:
    if device not in _default:
        _default[device] = Matcher(device)
    return _default[device]


class KeypointMatching:
    """Drop-in for ``ImageProcessing.KeypointMatching`` (KeypointMatching.cs:8-69).

    Parameterless like the reference's constructor (:10-12); ``device`` and
    ``desc_bits`` are optional extras (``desc_bits`` = ``NumGaussianPairs``,
    appsettings.json:23, default 256; widened automatically if a descriptor
    needs more bits).
    """

    def __init__(self, device: int = 0, desc_bits: int = 256):
        self._matcher = default_matcher(device)
        self._desc_bits = desc_bits

    def _pack(self, keypoints: Sequence[Keypoint], bits: int) -> np.ndarray:
        return pack_descriptors([int(k.BriefDescriptor if hasattr(k, "BriefDescriptor") else k.descriptor)
                                 for k in keypoints], bits)

    def MatchKeypoints(self, keypoints1: List[Keypoint], keypoints2: List[Keypoint]) -> List[KeypointPair]:
        bits = self._desc_bits
        for k in list(keypoints1) + list(keypoints2):
            d = int(k.BriefDescriptor if hasattr(k, "BriefDescriptor") else k.descriptor)
            if d < 0:
                raise ValueError("BriefDescriptor must be non-negative")
            bits = max(bits, d.bit_length())
        q, t = self._pack(keypoints1, bits), self._pack(keypoints2, bits)
        triples = self._matcher.match_greedy(q, t, bits, reference_compat_tail=True)
        return [KeypointPair(Keypoint1=keypoints1[i], Keypoint2=keypoints2[j], Distance=int(d))
                for i, j, d in triples.tolist()]


def match_keypoints(keypoints1, keypoints2, hamming_threshold: int = -1, device: int = 0) -> np.ndarray:
    """Drop-in for ``photogrammetry.image_processing.keypoint_matching.match_keypoints``
    (keypoint_matching.py:7-33): ``int64[len(k1), len(k2), 2]`` of ``(idx2, dist)`` with every row sorted
    by distance.  ``hamming_threshold`` is accepted and ignored, as upstream."""
    bits = 256
    d1 = [int(getattr(k, "descriptor", getattr(k, "BriefDescriptor", None))) for k in keypoints1]
    d2 = [int(getattr(k, "descriptor", getattr(k, "BriefDescriptor", None))) for k in keypoints2]
    for d in d1 + d2:
        bits = max(bits, d.bit_length())
    return default_matcher(device).match_keypoints_sorted(pack_descriptors(d1, bits), pack_descriptors(d2, bits), bits)


def match_keypoints_nearest(keypoints1, keypoints2, hamming_threshold: int = -1, device: int = 0):
    """Nearest-neighbour view of ``match_keypoints`` (keypoint_matching.py:7-33 +
    scripts/match_keypoints.py:121-134): for every keypoint of image 1 the
    nearest keypoint of image 2 and its distance, kept if
    ``hamming_threshold < 0 or dist <= hamming_threshold``.
    Returns ``int32[k, 3]`` rows (idx1, idx2, dist)."""
    bits = 256
    d1 = [int(getattr(k, "descriptor", getattr(k, "BriefDescriptor", None))) for k in keypoints1]
    d2 = [int(getattr(k, "descriptor", getattr(k, "BriefDescriptor", None))) for k in keypoints2]
    for d in d1 + d2:
        bits = max(bits, d.bit_length())
    m = default_matcher(device)
    return m.match_ratio_crosscheck(pack_descriptors(d1, bits), pack_descriptors(d2, bits), ratio=0.0,
                                    cross_check=False, max_dist=hamming_threshold, desc_bits=bits)
