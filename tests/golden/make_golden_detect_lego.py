#!/usr/bin/env python
"""Second golden vector for the keypoint producer, again made BY THE REFERENCE'S OWN PYTHON CODE, on a natural image:
a 720 x 960 crop of the two lego photographs the reference ships (data/feature_matching_test/lego_space_1_from_*.jpg;
the full 4000 x 3000 frames are out of reach of the reference's pure-Python detector).

    python tests/golden/make_golden_detect_lego.py [--reference /root/reference]      # build container only

Writes ``tests/golden/lego_crop_detect.npz`` with the same fields as star_detect.npz (make_golden_detect.py): gray0/1,
pairs (np.random.seed(7)), uv0/1, desc0/1, twin_nearest_dist, twin_sorted_dists.
"""
from __future__ import annotations

import argparse
import io
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
CROP = (slice(1600, 2320), slice(900, 1860))             # rows, columns


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    ap.add_argument("--threshold", type=int, default=25)
    args = ap.parse_args()
    ref = args.reference
    sys.path.insert(0, os.path.join(ref, "python_src"))
    import cv2
    from photogrammetry.image_processing.keypoint_detection import FASTKeypointDetector   # the reference's own
    from photogrammetry.image_processing.keypoint_matching import match_keypoints
    from photogrammetry.storage.image_db import ImageDB

    from photogrammetry_b200.descriptors import pack_descriptors

    data = os.path.join(ref, "data", "feature_matching_test")
    imgs = [np.ascontiguousarray(cv2.imread(os.path.join(data, f))[CROP])
            for f in ("lego_space_1_from_left.jpg", "lego_space_1_from_right.jpg")]
    h, w = imgs[0].shape[:2]
    db = ImageDB(h, w)
    ids = [db.add_image(im) for im in imgs]
    np.random.seed(7)
    det = FASTKeypointDetector(args.threshold, db)
    out = {"pairs": np.array(det._gaussian_pairs, dtype=np.int64), "threshold": np.int64(args.threshold)}
    kps = []
    for k, i in enumerate(ids):
        kp = det.detect_points(i)
        kps.append(kp)
        out[f"gray{k}"] = db.get_bw_image(i).astype(np.uint8)
        assert (out[f"gray{k}"].astype(np.int16) == db.get_bw_image(i)).all()
        out[f"uv{k}"] = np.array([p.coord for p in kp], dtype=np.int32).reshape(-1, 2)
        out[f"desc{k}"] = pack_descriptors([int(p.descriptor) for p in kp], 256)
        print(f"image {k}: {len(kp)} keypoints")
    twin = match_keypoints(kps[0], kps[1], -1)
    out["twin_nearest_dist"] = twin[:, 0, 1].astype(np.int64)
    out["twin_sorted_dists"] = twin[:, :, 1].astype(np.int16)
    # an .npz whose members are bzip2-compressed: np.load reads it like any other, and it stays under 1 MB where
    # np.savez_compressed (deflate) writes 1.2 MB
    with zipfile.ZipFile(os.path.join(HERE, "lego_crop_detect.npz"), "w", compression=zipfile.ZIP_BZIP2) as z:
        for k, v in out.items():
            buf = io.BytesIO()
            np.save(buf, v)
            z.writestr(f"{k}.npy", buf.getvalue())
    print("wrote lego_crop_detect.npz", {k: getattr(v, "shape", v) for k, v in out.items()})


if __name__ == "__main__":
    main()
