"""Host-side logic and the C-ABI surface (CPU: no compute calls)."""
import ctypes
import os
import re

import numpy as np
import pytest

import photogrammetry_b200 as pkg
from oracle import orc
from photogrammetry_b200 import _lib, synthetic
from photogrammetry_b200.descriptors import as_descriptor_rows, pack_descriptors, stride_for_bits, unpack_descriptors
from photogrammetry_b200.keypoint import Coordinate, Keypoint
from photogrammetry_b200.keypoint_cache import load_keypoint_dat, save_keypoint_dat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pack_roundtrip_and_layout():
    vals = [0, 1, (1 << 255) | 5, (1 << 256) - 1, 0x0102030405060708]
    rows = pack_descriptors(vals, 256)
    assert rows.shape == (5, 32) and rows.dtype == np.uint8
    assert unpack_descriptors(rows) == vals
    assert rows[4, :8].tolist() == [8, 7, 6, 5, 4, 3, 2, 1]          # little-endian, like BigInteger.ToByteArray
    assert stride_for_bits(1) == 16 and stride_for_bits(128) == 16 and stride_for_bits(129) == 32
    assert stride_for_bits(512) == 64
    with pytest.raises(ValueError):
        pack_descriptors([1 << 256], 256)
    with pytest.raises(ValueError):
        pack_descriptors([-1], 256)
    rows2, bits = as_descriptor_rows(np.zeros((3, 20), dtype=np.uint8))
    assert rows2.shape == (3, 32) and bits == 160


@pytest.mark.parametrize("bits", [1, 8, 100, 128, 130, 256, 512])
def test_synthetic_generators_match_oracle(bits):
    a = synthetic.uniform_descriptors(99, 37, bits)
    assert (a == orc.gen_uniform(99, 37, bits)).all()
    assert (synthetic.noisy_copy_descriptors(7, a, bits) == orc.gen_noisy_copy(7, a, bits)).all()
    if bits % 8:
        assert (np.bitwise_count(a[:, bits // 8]) <= bits % 8).all()   # bits >= desc_bits are zero


def test_config2_is_deterministic():
    q1, t1 = synthetic.config2_pair(256, "C")
    q2, t2 = synthetic.config2_pair(256, "C")
    assert (q1 == q2).all() and (t1 == t2).all()
    assert np.bitwise_count(q1).sum(axis=1).mean() == pytest.approx(128, abs=4)


def test_keypoint_cache_roundtrip(tmp_path):
    kps = [Keypoint(Coordinate(3, 4), 12345678901234567890), Keypoint(Coordinate(0, 9), (1 << 255) + 7)]
    p = tmp_path / "x.dat"
    save_keypoint_dat(str(p), kps)
    back = load_keypoint_dat(str(p))
    assert [k.BriefDescriptor for k in back] == [k.BriefDescriptor for k in kps]
    assert [k.coord for k in back] == [(3, 4), (0, 9)]


def test_keypoint_cache_refuses_code_execution(tmp_path):
    """A crafted cache file must not reach builtins.eval / os.system through REDUCE (exact-name whitelist)."""
    import pickle
    for payload in (b"cbuiltins\neval\n(V1+1\ntR.", b"cos\nsystem\n(Vtrue\ntR.", b"cnumpy\nload\n(Vx\ntR."):
        path = tmp_path / "evil.dat"
        path.write_bytes(payload)
        with pytest.raises(pickle.UnpicklingError):
            load_keypoint_dat(str(path))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "pgmatch.h")).read()
    declared = sorted(set(re.findall(r"\b(pgm_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no prototypes found in include/pgmatch.h"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"libpgmatch.so does not export {name}"
    assert lib.pgm_version() == 100
    assert b"no CPU fallback" in lib.pgm_status_string(_lib.PGM_E_NO_DEVICE)


def test_stats_struct_matches_header():
    header = open(os.path.join(ROOT, "include", "pgmatch.h")).read()
    body = header[header.index("typedef struct pgm_stats {"):header.index("} pgm_stats;")]
    fields = re.findall(r"int(?:32|64)_t\s+(\w+);", body)
    assert fields == [n for n, _ in _lib.Stats._fields_]
    assert ctypes.sizeof(_lib.Stats) == 4 * 4 + 5 * 8


def test_product_never_imports_the_oracle():
    pkg_dir = os.path.dirname(pkg.__file__)
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "liborc" not in src and "pgm_oracle" not in src, f


def test_every_environment_variable_the_library_reads_is_documented():
    """The library's getenv names are exactly the INTEGRATION.md section 5 table (PGM_LIB is read by the Python side)."""
    csrc = os.path.join(ROOT, "photogrammetry_b200", "csrc")
    read = set()
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh", ".h")):
            read |= set(re.findall(r'getenv\(\s*"(PGM_[A-Z0-9_]+)"', open(os.path.join(csrc, f)).read()))
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    section = doc.split("## 5. Diagnostics", 1)[1].split("\n## ", 1)[0]
    documented = {m for line in section.splitlines() if line.startswith("| `PGM_")
                  for m in re.findall(r"`(PGM_[A-Z0-9_]+)", line.split("|")[1])}
    assert read, "no getenv calls found"
    assert read == documented - {"PGM_LIB"}, (sorted(read - documented), sorted(documented - read - {"PGM_LIB"}))


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from photogrammetry_b200.keypoint_matching import KeypointMatching, Matcher
    with pytest.raises(_lib.PgmatchLibraryError):
        Matcher(0)
    with pytest.raises(_lib.PgmatchLibraryError):
        KeypointMatching()


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The boundary is a C ABI: include/pgmatch.h must compile as C99 and a C program must link and run against
    libpgmatch.so (what a P/Invoke / cgo / JNI shim does).  Without a GPU pgm_create has to refuse, loudly."""
    import shutil
    import subprocess
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        pytest.skip("no C compiler")
    libdir = os.path.dirname(_lib.LIB_PATH)
    src = tmp_path / "consumer.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "pgmatch.h"
int main(void) {
    pgm_handle *h = NULL;
    int rc;
    if (pgm_version() != 100) return 10;
    if (!strstr(pgm_status_string(PGM_E_NO_DEVICE), "no CPU fallback")) return 11;
    rc = pgm_create(0, &h);
    if (rc == PGM_OK) {                       /* a B200 is present: one tiny call through the ABI */
        unsigned char q[32] = {0}, t[64] = {0};
        int32_t qi[1], tj[1], dd[1], cnt = 0;
        t[32] = 1;                            /* train row 1 differs from the query in one bit */
        rc = pgm_match_hamming_greedy(h, q, 1, t, 2, 256, 32, qi, tj, dd, 1, &cnt, PGM_FLAG_REFERENCE_COMPAT_TAIL);
        if (rc != PGM_OK || cnt != 1 || qi[0] != 0 || tj[0] != 0 || dd[0] != 0) return 12;
        pgm_destroy(h);
        puts("gpu");
    } else {
        if (rc != PGM_E_NO_DEVICE || h != NULL) return 13;
        puts("no-device");
    }
    return 0;
}
''')
    exe = tmp_path / "consumer"
    subprocess.run([cc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    str(src), "-o", str(exe), "-L", libdir, "-lpgmatch", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert out.stdout.strip() in ("gpu", "no-device")
