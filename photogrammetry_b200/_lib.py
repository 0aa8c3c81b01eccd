"""ctypes loader for libpgmatch.so (the C ABI declared in include/pgmatch.h).

The product path has NO CPU fallback: if the shared library is missing, or it
cannot create a handle because no sm_100 device is present, the error is raised
to the caller.  The oracle under ``oracle/`` is test infrastructure and is never
imported from here.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PGM_LIB") or os.path.join(_HERE, "libpgmatch.so")     # PGM_LIB: e.g. the bounds-checked build
CSRC_DIR = os.path.join(_HERE, "csrc")

PGM_OK = 0
PGM_E_INVALID_ARG = -1
PGM_E_CAPACITY = -2
PGM_E_CUDA = -3
PGM_E_NCCL = -4
PGM_E_EMPTY_TRAIN = -5
PGM_E_NOMEM = -6
PGM_E_NO_DEVICE = -7
PGM_FLAG_REFERENCE_COMPAT_TAIL = 0x1
PGM_FLAG_PYTHON_GENERATION = 0x2
PGM_FLAG_RANSAC_RANK_TEST = 0x4
PGM_TAIL_DISTANCE = 2147483647

# every symbol include/pgmatch.h declares (tests check the .so exports them all)
EXPORTED_SYMBOLS = (
    "pgm_version", "pgm_status_string", "pgm_create", "pgm_destroy", "pgm_last_error",
    "pgm_set_stream", "pgm_synchronize", "pgm_get_stats", "pgm_host_alloc", "pgm_host_free",
    "pgm_match_hamming_greedy", "pgm_match_hamming_greedy_dev",
    "pgm_match_pairs_batch", "pgm_match_pairs_batch_dev",
    "pgm_knn2_hamming", "pgm_knn2_hamming_dev", "pgm_match_ratio_crosscheck", "pgm_match_ratio_crosscheck_batch_dev",
    "pgm_match_ratio_crosscheck_pairs_batch_dev", "pgm_pack_top2_keys_dev", "pgm_merge_top2_dev", "pgm_ratio_crosscheck_filter_dev",
    "pgm_match_keypoints_sorted", "pgm_match_keypoints_sorted_dev", "pgm_knn2_l2", "pgm_knn2_l2_dev", "pgm_l2_last_fallback_rows",
    "pgm_knn2_l2_pairs_batch_dev", "pgm_match_l2_ratio_crosscheck_pairs_batch_dev",
    "pgm_fast_detect", "pgm_brief_describe", "pgm_nms", "pgm_detect_describe_dev", "pgm_detect_describe_batch_dev",
    "pgm_detect_nms_describe_batch_dev", "pgm_detect_describe_images_batch_dev",
    "pgm_ransac_score", "pgm_ransac_fundamental_pairs_batch_dev",
    "pgm_shard_create", "pgm_shard_edge_capacity", "pgm_shard_round", "pgm_shard_commit", "pgm_shard_finish_round",
    "pgm_shard_finish", "pgm_shard_destroy",
    "pgm_multi_unique_id", "pgm_multi_create", "pgm_multi_destroy", "pgm_multi_match_train_sharded_dev",
    "pgm_multi_knn2_train_sharded_dev", "pgm_multi_get_exchange",
    "pgm_set_profiling", "pgm_get_round_profile", "pgm_measure_popc_peak",
)


class PgmatchLibraryError(RuntimeError):
    """libpgmatch.so is missing/unloadable, or no usable B200 is present."""


class PgmatchError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"pgmatch status {status}: {message}")
        self.status = status


class EmptyTrainError(PgmatchError, IndexError):
    """Mirror of the ArgumentOutOfRangeException the reference throws at
    KeypointMatching.cs:61 (``keypoints2[0]`` on an empty list)."""


class Stats(C.Structure):
    _fields_ = [
        ("rounds", C.c_int32), ("kernel_launches", C.c_int32), ("host_syncs", C.c_int32), ("pairs", C.c_int32),
        ("distance_evals", C.c_int64), ("evals_computed", C.c_int64), ("matched", C.c_int64),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
    ]

    def as_dict(self) -> dict:
        return {name: int(getattr(self, name)) for name, _ in self._fields_}


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a into photogrammetry_b200/libpgmatch.so (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC_DIR, f) for f in os.listdir(CSRC_DIR) if f.endswith((".cu", ".cuh"))]
    srcs.append(os.path.join(os.path.dirname(_HERE), "include", "pgmatch.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", CSRC_DIR, "--no-print-directory"] + (["-B"] if force else [])
        subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


_lib = None
_lib_lock = threading.Lock()


def load() -> C.CDLL:
    """Load libpgmatch.so and declare prototypes.  Raises PgmatchLibraryError if it is missing."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise PgmatchLibraryError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C photogrammetry_b200/csrc`.  There is no CPU fallback.")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover
            raise PgmatchLibraryError(f"cannot load {LIB_PATH}: {e}") from e
        u8p, i32p, i64p, vp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p   # raw addresses: host or device
        lib.pgm_version.restype = C.c_int
        lib.pgm_status_string.restype = C.c_char_p
        lib.pgm_status_string.argtypes = [C.c_int]
        lib.pgm_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.pgm_destroy.argtypes = [C.c_void_p]
        lib.pgm_last_error.restype = C.c_char_p
        lib.pgm_last_error.argtypes = [C.c_void_p]
        lib.pgm_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        lib.pgm_synchronize.argtypes = [C.c_void_p]
        lib.pgm_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
        lib.pgm_host_free.argtypes = [C.c_void_p]
        lib.pgm_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        greedy = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32, i32p, i32p, i32p,
                  C.c_int32, C.POINTER(C.c_int32), C.c_uint32]
        lib.pgm_match_hamming_greedy.argtypes = greedy
        lib.pgm_match_hamming_greedy_dev.argtypes = greedy
        batch = [C.c_void_p, u8p, i64p, C.c_int32, i32p, C.c_int32, C.c_int32, C.c_int32, i32p, i32p, i32p,
                 C.c_int64, i32p, C.c_uint32]
        lib.pgm_match_pairs_batch.argtypes = batch
        lib.pgm_match_pairs_batch_dev.argtypes = batch
        knn = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32, i32p, i32p, i32p, i32p]
        lib.pgm_knn2_hamming.argtypes = knn
        lib.pgm_knn2_hamming_dev.argtypes = knn
        lib.pgm_pack_top2_keys_dev.argtypes = [C.c_void_p, i32p, i32p, i32p, i32p, C.c_int32, C.c_int32, i32p]
        lib.pgm_merge_top2_dev.argtypes = [C.c_void_p, i32p, C.c_int32, C.c_int32, i32p, i32p, i32p, i32p]
        lib.pgm_ratio_crosscheck_filter_dev.argtypes = [C.c_void_p, C.c_int32, C.c_int32, i32p, i32p, i32p, i32p,
                                                        C.c_float, C.c_int32, C.c_int32, i32p, i32p, i32p,
                                                        C.POINTER(C.c_int32)]
        lib.pgm_match_keypoints_sorted.argtypes = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32, i64p]
        lib.pgm_match_keypoints_sorted_dev.argtypes = lib.pgm_match_keypoints_sorted.argtypes
        lib.pgm_knn2_l2.argtypes = [C.c_void_p, vp, C.c_int32, vp, C.c_int32, C.c_int32, i32p, vp, i32p, vp]
        lib.pgm_knn2_l2_dev.argtypes = [C.c_void_p, vp, C.c_int32, vp, C.c_int32, C.c_int32, i32p, vp, i32p, vp, vp]
        lib.pgm_l2_last_fallback_rows.argtypes = [C.c_void_p]
        lib.pgm_knn2_l2_pairs_batch_dev.argtypes = [C.c_void_p, vp, i64p, C.c_int32, i32p, C.c_int32, C.c_int32, i32p, vp, i32p,
                                                    vp, C.c_int64]
        lib.pgm_match_l2_ratio_crosscheck_pairs_batch_dev.argtypes = [C.c_void_p, vp, i64p, C.c_int32, i32p, C.c_int32,
                                                                      C.c_int32, C.c_float, C.c_int32, C.c_float, i32p, i32p,
                                                                      vp, C.c_int64, i32p]
        lib.pgm_match_ratio_crosscheck.argtypes = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32,
                                                   C.c_float, C.c_int32, C.c_int32, i32p, i32p, i32p, C.c_int32,
                                                   C.POINTER(C.c_int32)]
        lib.pgm_match_ratio_crosscheck_batch_dev.argtypes = [C.c_void_p, u8p, i64p, C.c_int32, i32p, C.c_int32, C.c_int32,
                                                             C.c_int32, C.c_float, C.c_int32, C.c_int32, i32p, i32p, i32p,
                                                             C.c_int64, i32p]
        lib.pgm_match_ratio_crosscheck_pairs_batch_dev.argtypes = lib.pgm_match_ratio_crosscheck_batch_dev.argtypes
        lib.pgm_fast_detect.argtypes = [C.c_void_p, vp, C.c_int32, C.c_int32, C.c_float, C.c_uint32, i32p, i32p,
                                        C.c_int32, C.POINTER(C.c_int32)]
        lib.pgm_brief_describe.argtypes = [C.c_void_p, vp, C.c_int32, C.c_int32, i32p, C.c_int32, i32p, C.c_int32,
                                           C.c_int32, C.c_uint32, u8p]
        lib.pgm_nms.argtypes = [C.c_void_p, i32p, i32p, C.c_int32, C.c_int32, i32p, C.POINTER(C.c_int32)]
        lib.pgm_detect_describe_dev.argtypes = [C.c_void_p, vp, C.c_int32, C.c_int32, C.c_float, C.c_int32, i32p, C.c_int32,
                                                C.c_int32, C.c_uint32, i32p, i32p, u8p, C.c_int32, C.POINTER(C.c_int32)]
        lib.pgm_detect_describe_batch_dev.argtypes = [C.c_void_p, vp, C.c_int32, C.c_int32, C.c_int32, C.c_float, i32p,
                                                      C.c_int32, C.c_int32, C.c_uint32, i32p, i32p, u8p, C.c_int32, i32p,
                                                      i32p]
        lib.pgm_detect_nms_describe_batch_dev.argtypes = [C.c_void_p, vp, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                                          C.c_int32, i32p, C.c_int32, C.c_int32, C.c_uint32, i32p, i32p,
                                                          u8p, C.c_int32, i32p, i32p]
        lib.pgm_detect_describe_images_batch_dev.argtypes = [C.c_void_p, vp, i64p, i32p, i32p, C.c_int32, C.c_float,
                                                             C.c_int32, i32p, C.c_int32, C.c_int32, C.c_uint32, i32p,
                                                             i32p, u8p, C.c_int32, i32p, i32p]
        lib.pgm_ransac_score.argtypes = [C.c_void_p, vp, u8p, C.c_int32, i32p, i32p, C.c_int32, C.c_float, i32p,
                                         C.POINTER(C.c_int32), u8p]
        lib.pgm_ransac_fundamental_pairs_batch_dev.argtypes = [C.c_void_p, i32p, i64p, C.c_int32, i32p, C.c_int32, i32p, i32p,
                                                               i64p, i32p, C.c_int32, C.c_int32, C.c_float, C.c_uint64,
                                                               C.c_uint32, i32p, i32p, vp, u8p, C.c_int64, vp, i32p]
        lib.pgm_shard_create.argtypes = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.POINTER(C.c_void_p)]
        lib.pgm_shard_round.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
        lib.pgm_shard_commit.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]
        lib.pgm_shard_edge_capacity.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]
        lib.pgm_shard_finish_round.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                                               C.POINTER(C.c_int32)]
        lib.pgm_multi_unique_id.argtypes = [C.c_void_p]
        lib.pgm_multi_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
        lib.pgm_multi_destroy.argtypes = [C.c_void_p]
        lib.pgm_multi_match_train_sharded_dev.argtypes = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32,
                                                          C.c_int32, C.c_int32, i32p, i32p, i32p, C.c_int32,
                                                          C.POINTER(C.c_int32), C.c_uint32, C.POINTER(C.c_int32)]
        lib.pgm_multi_knn2_train_sharded_dev.argtypes = [C.c_void_p, u8p, C.c_int32, u8p, C.c_int32, C.c_int32, C.c_int32,
                                                         C.c_int32, i32p, i32p, i32p, i32p]
        lib.pgm_multi_get_exchange.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
        lib.pgm_shard_finish.argtypes = [C.c_void_p, i32p, i32p, i32p, C.c_uint32, C.POINTER(C.c_int32),
                                         C.POINTER(C.c_int32)]
        lib.pgm_shard_destroy.argtypes = [C.c_void_p]
        lib.pgm_set_profiling.argtypes = [C.c_void_p, C.c_int32]
        lib.pgm_get_round_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
        lib.pgm_measure_popc_peak.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        _ = vp
        _lib = lib
        return _lib


class _PinnedBlock:
    """Owner of one pgm_host_alloc block; numpy arrays made from it keep it alive through ``.base``."""

    def __init__(self, nbytes: int):
        self._lib = load()
        self.ptr = C.c_void_p()
        rc = self._lib.pgm_host_alloc(max(int(nbytes), 1), C.byref(self.ptr))
        if rc != PGM_OK or not self.ptr.value:
            raise PgmatchLibraryError(f"pgm_host_alloc({nbytes}) failed: {self._lib.pgm_status_string(rc).decode()}")
        self.nbytes = max(int(nbytes), 1)

    def __del__(self):  # pragma: no cover
        try:
            if self.ptr and self.ptr.value:
                self._lib.pgm_host_free(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


def pinned_empty(shape, dtype):
    """A numpy array in page-locked host memory (pgm_host_alloc): the host-buffer entry points copy to and from
    such arrays directly, without their internal staging pass."""
    import numpy as np
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
    block = _PinnedBlock(n * dt.itemsize)
    buf = (C.c_char * block.nbytes).from_address(block.ptr.value)
    buf._pgm_owner = block                       # ties the allocation's lifetime to the ctypes buffer
    return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)


def status_string(status: int) -> str:
    return load().pgm_status_string(status).decode()
