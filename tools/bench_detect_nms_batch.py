#!/usr/bin/env python
"""Batched detect -> NMS -> BRIEF (pgm_detect_nms_describe_batch_dev) against a loop of pgm_detect_describe_dev over the
same frames, on one GPU.

    python tools/bench_detect_nms_batch.py [--reps 30 --out profiles/x.json]

Workloads:
  star32      the 32-frame shifted-star sequence (BASELINE configs[2]) on the C# scale (Grayscale.K), threshold 0.1, r = 10
  large8      8 frames of 3000 x 4000 (synthetic.rectangles_image, tools/detect_one.py's image), frame k shifted by
              150 k px, threshold 0.1, r = 10
  chain       the dotted-row frame (synthetic.dotted_row_image): 496 keypoints whose parallel NMS rounds form a chain
              of 496, r = 4
For each: ms per batch for both forms (host clock around the call, ended by a device synchronise; median of --reps
after one warm-up of each form, the two forms alternating), host_syncs and kernel_launches of both forms (summed
over the loop's calls), FAST keypoints and survivors per frame, and whether both forms give the same xy, scores and
descriptor bytes.  The card's name, power limit and max SM clock are read in the same run (read-only nvidia-smi
query).  The frames stay on the device; the 8 large frames (384 MB) exceed the L2, the others fit in it."""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from oracle import detect_np as D
from photogrammetry_b200 import keypoint_detection as kd
from photogrammetry_b200 import sequence, synthetic
from photogrammetry_b200.keypoint_matching import Matcher

TABLE = D.gaussian_pairs(11, 256, 50).reshape(-1, 4).astype(np.int32)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in out[0].split(","))))
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


def workloads():
    star = sequence.shifted_frames(sequence.star_gray(), 32, 5)
    yield "star32", np.stack([kd.grayscale_from_rgb8(np.repeat(f[..., None], 3, axis=2)) for f in star]), 0.1, 10, 4096
    yield "large8", np.stack([synthetic.rectangles_image(shift=150 * k) for k in range(8)]), 0.1, 10, 8192
    yield "chain", synthetic.dotted_row_image()[None], 0.1, 4, 4096


def run_batch(m, d, th, r, cap):
    out = m.detect_describe_batch_dev(d, th, TABLE, capacity=cap, nms_radius=r)
    torch.cuda.synchronize()
    st = m.stats()
    return out, {"host_syncs": st["host_syncs"], "kernel_launches": st["kernel_launches"]}


def run_loop(m, d, th, r, cap):
    outs, syncs, launches = [], 0, 0
    for k in range(d.shape[0]):
        outs.append(m.detect_describe_dev(d[k], th, TABLE, nms_radius=r, capacity=cap))
        st = m.stats()
        syncs += st["host_syncs"]; launches += st["kernel_launches"]
    torch.cuda.synchronize()
    return outs, {"host_syncs": syncs, "kernel_launches": launches}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3        # fn ends in a device synchronise


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    m = Matcher(0)
    res = {"gpu": gpu_info(), "reps": a.reps, "workloads": {}}
    for name, frames, th, r, cap in workloads():
        d = torch.from_numpy(frames).cuda()
        fast = m.detect_describe_batch_dev(d, th, TABLE, capacity=1)[3]     # without NMS: the FAST totals
        (xy, sc, desc, counts), bstats = run_batch(m, d, th, r, cap)
        loop, lstats = run_loop(m, d, th, r, cap)
        equal = all(int(counts[k]) == len(lx) and torch.equal(xy[k, :len(lx)], lx) and torch.equal(sc[k, :len(lx)], ls)
                    and torch.equal(desc[k, :len(lx)], ld) for k, (lx, ls, ld) in enumerate(loop))
        tb, tl = [], []
        for _ in range(a.reps):
            tb.append(timed(lambda: run_batch(m, d, th, r, cap)))
            tl.append(timed(lambda: run_loop(m, d, th, r, cap)))
        res["workloads"][name] = {
            "frames": int(d.shape[0]), "height": int(d.shape[1]), "width": int(d.shape[2]), "threshold": th, "radius": r,
            "fast_keypoints": [int(x) for x in fast], "survivors": [int(x) for x in counts],
            "batch_ms_median": float(np.median(tb)), "loop_ms_median": float(np.median(tl)),
            "batch_ms_min": float(np.min(tb)), "loop_ms_min": float(np.min(tl)),
            "batch_stats": bstats, "loop_stats": lstats, "outputs_equal": bool(equal)}
        print(name, json.dumps(res["workloads"][name]), flush=True)
        del d
    m.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
