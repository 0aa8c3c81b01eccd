#!/usr/bin/env python
"""Detect -> (NMS) -> BRIEF for images of different sizes in one call (pgm_detect_describe_images_batch_dev), on one GPU.

    python tools/bench_detect_images_batch.py [--reps 20 --parent-tree DIR --out profiles/x.json]

--parent-tree: a checkout of the parent commit with its library built (photogrammetry_b200/libpgmatch.so).

Workloads (threshold 0.1 on the C# scale, BRIEF-256):
  (a) mixed16   16 images alternating 4000 x 3000 and 3000 x 4000 (synthetic.rectangles_image, seeds 0..15), r = 10
                and no NMS: the call against a loop of pgm_detect_describe_dev, with time, host syncs and launches
  (b) skewed    one 4000 x 3000 image and 63 of 640 x 480: the call against the same images as two uniform batch
                calls (one per size), which is what a grid with no idle CTAs costs, and against the loop
  (c) uniform   the r05 workloads of pgm_detect_nms_describe_batch_dev (32 star frames r = 10, 8 frames of 4000 x 3000
                r = 10, the dotted-row chain r = 4) and pgm_detect_describe_batch_dev on the 8 large frames, timed with
                this tree's library and the parent commit's (--parent-tree, its package and its library, selected by
                PGM_LIB), the two alternating in separate processes
  (d) chain     image_set.match_image_set_dev on (a)'s 16 images with r = 10, all 120 pairs, greedy: ms per stage
Times are host clocks around work that ends in a device synchronise, medians of --reps after a warm-up, the compared
forms alternating.  Outputs of compared forms are compared in the same run.  The card's name, power limit and max SM
clock are read in the same run (read-only nvidia-smi query).  The 16 large images (768 MB) exceed the L2."""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

TH = 0.1


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in out[0].split(","))))
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


def table():
    from oracle import detect_np as D
    return D.gaussian_pairs(11, 256, 50).reshape(-1, 4).astype(np.int32)


def timed(fn, m):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    st = m.stats()
    return out, (time.perf_counter() - t0) * 1e3, st


def call_set(m, ims, r, cap):
    return lambda: m.detect_describe_images_batch_dev(ims, TH, TABLE, capacity=cap, nms_radius=r)


def call_loop(m, ims, r, cap):
    def run():
        outs, syncs, launches = [], 0, 0
        for im in ims:
            outs.append(m.detect_describe_dev(im, TH, TABLE, nms_radius=r, capacity=cap))
            st = m.stats()
            syncs += st["host_syncs"]; launches += st["kernel_launches"]
        return outs, syncs, launches
    return run


def same(set_out, loop_outs):
    xy, sc, desc, counts = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in set_out)
    for k, (exy, esc, edesc) in enumerate(loop_outs):
        n = len(exy)
        if int(counts[k]) != n or not ((xy[k, :n] == exy.cpu().numpy()).all() and (sc[k, :n] == esc.cpu().numpy()).all()
                                       and (desc[k, :n] == edesc.cpu().numpy()).all()):
            return False
    return True


def compare(m, ims, r, cap, reps, extra=None):
    """the set call against the loop (and `extra`: name -> (fn, combine)), alternating; medians"""
    fs = {"set": call_set(m, ims, r, cap), "loop": call_loop(m, ims, r, cap)}
    fs.update(extra or {})
    times = {k: [] for k in fs}
    last = {}
    for rep in range(reps + 1):
        for name, fn in fs.items():
            out, ms, st = timed(fn, m)
            if rep:
                times[name].append(ms)
            last[name] = (out, st)
    set_out, set_st = last["set"]
    loop_out, loop_syncs, loop_launches = last["loop"][0]
    res = {"r": r, "ms_set": float(np.median(times["set"])), "ms_loop": float(np.median(times["loop"])),
           "syncs_set": set_st["host_syncs"], "launches_set": set_st["kernel_launches"],
           "syncs_loop": loop_syncs, "launches_loop": loop_launches,
           "counts": [int(x) for x in set_out[3]][:4], "total_keypoints": int(np.sum(set_out[3])),
           "equal_outputs": same(set_out, loop_out)}
    for name in (extra or {}):
        res["ms_" + name] = float(np.median(times[name]))
    return res


def mixed16():
    from photogrammetry_b200 import synthetic
    return [synthetic.rectangles_image(3000, 4000, seed=k) if k % 2 == 0 else synthetic.rectangles_image(4000, 3000, seed=k)
            for k in range(16)]


def child_uniform(reps):
    """(c) in this process's library: ms per call of each uniform workload, printed as one JSON line"""
    import torch
    from photogrammetry_b200 import keypoint_detection as kd
    from photogrammetry_b200 import sequence, synthetic
    from photogrammetry_b200.keypoint_matching import Matcher
    star = sequence.shifted_frames(sequence.star_gray(), 32, 5)
    loads = {"star32_r10": (np.stack([kd.grayscale_from_rgb8(np.repeat(f[..., None], 3, axis=2)) for f in star]), 10, 4096),
             "large8_r10": (np.stack([synthetic.rectangles_image(shift=150 * k) for k in range(8)]), 10, 8192),
             "chain_r4": (synthetic.dotted_row_image()[None], 4, 4096),
             "large8_no_nms": (None, -1, 65536)}
    loads["large8_no_nms"] = (loads["large8_r10"][0], -1, 65536)
    out = {}
    with Matcher(0) as m:
        for name, (frames, r, cap) in loads.items():
            d = torch.from_numpy(frames).cuda()
            ts, res = [], None
            for rep in range(reps + 1):
                res, ms, st = timed(lambda: m.detect_describe_batch_dev(d, TH, TABLE, capacity=cap, nms_radius=r), m)
                if rep:
                    ts.append(ms)
            xy, sc, desc, counts = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in res)
            written = np.arange(cap)[None, :] < np.minimum(counts, cap)[:, None]      # slots past a count are unwritten
            out[name] = {"ms": ts, "syncs": st["host_syncs"], "launches": st["kernel_launches"],
                         "counts_sum": int(np.sum(counts)), "xy_sum": int(xy[written].astype(np.int64).sum()),
                         "sc_sum": int(sc[written].astype(np.int64).sum()),
                         "desc_xor": int(np.bitwise_xor.reduce(desc[written].view(np.uint64).ravel()))}
    print("CHILD " + json.dumps(out))


def uniform_ab(parent_tree, rounds, reps):
    trees = {"branch": ROOT, "parent": os.path.abspath(parent_tree)}
    runs = {k: [] for k in trees}
    for _ in range(rounds):
        for name, tree in trees.items():
            env = dict(os.environ, PGM_LIB=os.path.join(tree, "photogrammetry_b200", "libpgmatch.so"))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", tree, "--reps", str(reps)], env=env,
                               capture_output=True, text=True, timeout=1800)
            line = [x for x in p.stdout.splitlines() if x.startswith("CHILD ")]
            if not line:
                raise RuntimeError(f"{name}: {p.stderr[-2000:]}")
            runs[name].append(json.loads(line[0][6:]))
    res = {}
    for w in runs["branch"][0]:
        b = [t for r in runs["branch"] for t in r[w]["ms"]]
        pa = [t for r in runs["parent"] for t in r[w]["ms"]]
        per_round = {k: [float(np.median(r[w]["ms"])) for r in runs[k]] for k in runs}
        keys = ("syncs", "launches", "counts_sum", "xy_sum", "sc_sum", "desc_xor")
        res[w] = {"ms_branch": float(np.median(b)), "ms_parent": float(np.median(pa)),
                  "round_medians_branch": per_round["branch"], "round_medians_parent": per_round["parent"],
                  "syncs_launches_branch": [runs["branch"][0][w]["syncs"], runs["branch"][0][w]["launches"]],
                  "syncs_launches_parent": [runs["parent"][0][w]["syncs"], runs["parent"][0][w]["launches"]],
                  "equal_outputs": all(runs["branch"][0][w][k] == runs["parent"][0][w][k] for k in keys)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)     # (c): the tree whose package is timed
    a = ap.parse_args()
    if a.child:
        sys.path.insert(0, a.child)
        child_uniform(a.reps)
        return
    import torch
    from photogrammetry_b200 import image_set, synthetic
    from photogrammetry_b200.keypoint_matching import Matcher
    res = {"gpu": gpu_info(), "reps": a.reps}
    with Matcher(0) as m:
        ims = [torch.from_numpy(x).cuda() for x in mixed16()]
        res["a_mixed16"] = [compare(m, ims, r, 65536, a.reps) for r in (10, -1)]
        print(json.dumps(res["a_mixed16"]), flush=True)

        big = torch.from_numpy(synthetic.rectangles_image(3000, 4000, seed=1)).cuda()
        small = torch.from_numpy(np.stack([synthetic.rectangles_image(480, 640, seed=100 + k) for k in range(63)])).cuda()
        skew = [big] + list(small)
        res["b_skewed"] = []
        for r in (10, -1):
            cap = 65536
            def two_uniform(r=r, cap=cap):
                m.detect_describe_batch_dev(big[None], TH, TABLE, capacity=cap, nms_radius=r)
                st1 = m.stats()
                m.detect_describe_batch_dev(small, TH, TABLE, capacity=cap, nms_radius=r)
                return st1
            res["b_skewed"].append(compare(m, skew, r, cap, a.reps, {"two_uniform_calls": two_uniform}))
        print(json.dumps(res["b_skewed"]), flush=True)

        stages = {k: [] for k in ("detect_ms", "compaction_ms", "match_ms", "ransac_ms", "total_ms")}
        for rep in range(min(a.reps, 10) + 1):
            tm = {}
            t0 = time.perf_counter()
            out = image_set.match_image_set_dev(m, ims, TH, TABLE, nms_radius=10, timings=tm)
            torch.cuda.synchronize()
            tm["total_ms"] = (time.perf_counter() - t0) * 1e3
            if rep:
                for k in stages:
                    stages[k].append(tm[k])
        res["d_chain"] = {"images": 16, "pairs": int(len(out.pair_list)), "method": "greedy", "nms_radius": 10,
                          "keypoints_per_image": [int(x) for x in out.counts],
                          "matches": int(np.sum(out.match_counts)),
                          "pairs_with_winner": int((out.best.cpu().numpy() >= 0).sum()),
                          **{k: float(np.median(v)) for k, v in stages.items()}}
        print(json.dumps(res["d_chain"]), flush=True)
        del ims, big, small, skew
    if a.parent_tree:
        res["c_uniform_ab"] = uniform_ab(a.parent_tree, a.rounds, a.reps)
        print(json.dumps(res["c_uniform_ab"]), flush=True)
    else:
        res["c_uniform_ab"] = "not measured (no --parent-tree)"
    res["gpu_after"] = gpu_info()
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    TABLE = table()
    main()
