#!/usr/bin/env python
"""Batched fundamental-matrix RANSAC (pgm_ransac_fundamental_pairs_batch_dev) on one GPU.

    python tools/bench_ransac_pairs.py [--pairs 10000 --per 512 --samples 2000 --out profiles/x.json]

One JSON line:
  configs2_chain  the K = 32 star sequence (BASELINE configs[2]): detect_describe_batch_dev -> match_ratio_crosscheck_batch_dev
                  -> this call on the 31 consecutive pairs (upstream's 2000 samples of 32, threshold 0.001, rank gate on);
                  ms per stage, best of --reps, each stage ended by a device synchronise
  synthetic       --pairs seeded two-view match lists (synthetic.two_view_matches: projections rounded to pixels, 30 %
                  outliers, --per matches each) at S = --samples, P = 32: call time (CUDA events, best of --reps after a
                  warm-up call), hypotheses/s, residuals/s (sum over pairs of count * S) and the residual loop's share of
                  the FP32 pipe, with the rank gate on (upstream) and off
  kernel_split_ms device time per kernel of one synthetic call (torch.profiler, a run of its own)
  gpu             name, power limit and max SM clock (read-only nvidia-smi query in the same run)

Share of peak: a residual is 16 FP32-pipe operations -- residual() is 3 x (2 FMUL + 2 FADD) for F . (x2, y2, 1) and
2 FMUL + 2 FADD for the dot product, no FMA contraction; the comparison and the counter are not counted -- against
148 SM x 128 FP32 lanes x the card's max SM clock, computed here and not a data-sheet figure.  The numerator is the
score loop's work only, the denominator the whole call (fp64 estimate and winner included): a call-level figure, not
a kernel's share of peak."""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from photogrammetry_b200 import sequence, synthetic
from photogrammetry_b200.keypoint_matching import Matcher
from photogrammetry_b200.sharding import consecutive_pairs

OPS_PER_RESIDUAL = 16


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in out[0].split(","))))
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


def chain(m, reps):
    frames = torch.from_numpy(sequence.shifted_frames(sequence.star_gray(), 32, 5).astype(np.float32)).cuda()
    table = sequence.pairs_table(sequence.star_pairs())
    plist = consecutive_pairs(32)
    best = None
    for _ in range(reps + 1):                                  # the first pass warms every shape up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        xy, _sc, desc, counts = m.detect_describe_batch_dev(frames, 50.0, table, capacity=4096, python_generation=True)
        offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        d_desc = torch.cat([desc[f, :int(counts[f])] for f in range(32)]).contiguous()
        d_xy = torch.cat([xy[f, :int(counts[f])] for f in range(32)]).contiguous()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        fo, fst, fcn = m.match_ratio_crosscheck_batch_dev(d_desc, offs, plist, 256, 0.8, True, -1)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        b, inl, F, mask = m.ransac_fundamental_pairs_batch_dev(d_xy, offs, plist, fo[0], fo[1], fst, fcn)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        ms = {"detect_describe_ms": (t1 - t0) * 1e3, "ratio_crosscheck_ms": (t2 - t1) * 1e3, "ransac_ms": (t3 - t2) * 1e3}
        if best is None or sum(ms.values()) < sum(best.values()):
            best = ms
    best["matches"] = int(fcn.sum())
    best["pairs_with_winner"] = int((b.cpu().numpy() >= 0).sum())
    return best


def timed(m, args, batch, rank, reps):
    xy, offs, pairs, qi, tj, st, cn = batch
    kw = dict(n_samples=args.samples, pairs_per_sample=32, threshold=0.001, seed=0, require_rank2=rank)
    m.ransac_fundamental_pairs_batch_dev(xy, offs, pairs, qi, tj, st, cn, **kw)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = m.ransac_fundamental_pairs_batch_dev(xy, offs, pairs, qi, tj, st, cn, **kw)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    return min(times), times, out


def kernel_split(m, args, batch):
    from torch.profiler import ProfilerActivity, profile
    xy, offs, pairs, qi, tj, st, cn = batch
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.ransac_fundamental_pairs_batch_dev(xy, offs, pairs, qi, tj, st, cn, n_samples=args.samples, require_rank2=True)
        torch.cuda.synchronize()
    split = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        for key in ("estimate_kernel", "pairs_score_kernel", "winner_kernel"):
            if key in e.key:
                split[key] = split.get(key, 0.0) + us * 1e-3
    return split


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10000)
    ap.add_argument("--per", type=int, default=512)
    ap.add_argument("--samples", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ransac_pairs.py measures on a GPU; there is none")
    info = gpu_info()
    m = Matcher(0)
    res = {"gpu": info, "configs2_chain": chain(m, args.reps)}
    xy, offs, pairs, qi, tj, st, cn = synthetic.two_view_matches(2024, args.pairs, args.per)
    batch = (torch.from_numpy(xy).cuda(), offs, pairs, torch.from_numpy(qi).cuda(), torch.from_numpy(tj).cuda(), st, cn)
    hyps = args.pairs * args.samples
    residuals = int(cn.astype(np.int64).sum()) * args.samples
    try:
        clock_hz = float(info["max_sm_clock"].split()[0]) * 1e6
    except Exception:
        clock_hz = None
    syn = {"pairs": args.pairs, "matches_per_pair": args.per, "samples": args.samples, "pairs_per_sample": 32,
           "hypotheses": hyps, "residuals": residuals}
    for rank in (True, False):
        t, times, out = timed(m, args, batch, rank, args.reps)
        row = {"seconds": t, "all_seconds": times, "hypotheses_per_s": hyps / t, "residuals_per_s": residuals / t,
               "pairs_with_winner": int((out[0].cpu().numpy() >= 0).sum())}
        if clock_hz:
            peak = 148 * 128 * clock_hz
            row["residual_fp32_ops_share_of_call"] = residuals * OPS_PER_RESIDUAL / t / peak
            row["peak_fp32_ops_per_s"] = peak
        syn["rank_test_on" if rank else "rank_test_off"] = row
    st_ = m.stats()
    syn["kernel_launches"], syn["host_syncs"] = st_["kernel_launches"], st_["host_syncs"]
    res["synthetic"] = syn
    res["kernel_split_ms"] = kernel_split(m, args, batch)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    m.close()


if __name__ == "__main__":
    main()
