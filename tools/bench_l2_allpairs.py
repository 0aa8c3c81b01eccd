#!/usr/bin/env python
"""Float descriptors, every pair of an image set in one call (pgm_knn2_l2_pairs_batch_dev and
pgm_match_l2_ratio_crosscheck_pairs_batch_dev), one GPU:

    python tools/bench_l2_allpairs.py [--images 512 --per 4096 --dim 128] [--out profiles/r04_l2_allpairs_1gpu.json]

One JSON line:
  knn2_job / ratio_job   all pairs a < b (130 816 at 512 images), device resident, alternated (A B A B); seconds,
                         distances/s, algorithmic fraction of the bf16 peak (2 D flops per distance, against the measured
                         1648.6 TFLOP/s DESIGN.md section 4.2 uses; the ratio job with cross-check computes every distance twice
                         and is charged for one)
  per_pair_loop          the same pairs' first --subset through a loop of pgm_knn2_l2_dev, alternated with the knn2 batch on
                         that subset in the same process; bit-identity of the subset's results
  single_32768           one 32 768 x 32 768 x D pgm_knn2_l2_dev call
  phases                 kernel time per phase (torch.profiler, CUDA activities) of one knn2 job and one ratio job in a
                         separate, profiled pass: conversion (l2b_prep + l2b_split16), GEMM, refinement, fallback, filter
  gpu                    name, power limit and max SM clock (read-only nvidia-smi query in the same run)
Descriptors: uniform [0, 1) floats, SIFT-like non-negative, image k from seed 5000 + k; the job's working set (1 GB of
descriptors, 2 GB of operands per chunk) exceeds the 126 MB L2."""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from photogrammetry_b200 import sharding
from photogrammetry_b200.keypoint_matching import Matcher

BF16_PEAK = 1648.6e12


def log(msg):
    print(f"[{time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


PHASES = {"conversion": ("l2b_prep_kernel", "l2b_split16_kernel"), "gemm": ("l2_topk_pair_kernel",),
          "refinement": ("l2b_refine_kernel",), "fallback": ("l2b_exact_rows_kernel",),
          "filter": ("l2b_filter_kernel", "l2b_scatter_kernel")}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return [dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(",")))) for line in out]
    except Exception as e:  # pragma: no cover
        return [{"error": str(e)}]


def phases(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {k: 0.0 for k in PHASES}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        for k, names in PHASES.items():
            if any(n in e.key for n in names):
                split[k] += us * 1e-3
    tot = sum(split.values())
    return {"kernel_ms": split, "share": {k: v / tot for k, v in split.items()} if tot else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--per", type=int, default=4096)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--subset", type=int, default=1024, help="pairs of the per-pair loop")
    ap.add_argument("--big", type=int, default=32768)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    n_img, per, dim = args.images, args.per, args.dim
    g = torch.Generator(device=dev)
    d_all = torch.empty((n_img * per, dim), dtype=torch.float32, device=dev)
    for k in range(n_img):
        g.manual_seed(5000 + k)
        d_all[k * per:(k + 1) * per] = torch.rand((per, dim), generator=g, device=dev)
    offs = np.arange(n_img + 1, dtype=np.int64) * per
    pairs = sharding.all_pairs(n_img)
    m = Matcher(0)
    evals = float(len(pairs)) * per * per

    def knn2(pl):
        r = m.knn2_l2_pairs_batch_dev(d_all, offs, pl)
        torch.cuda.synchronize()
        return r

    def ratio(pl):
        r = m.match_l2_ratio_crosscheck_pairs_batch_dev(d_all, offs, pl, 0.8, True)
        torch.cuda.synchronize()
        return r

    log("descriptors ready")
    warm = pairs[:256]
    knn2(warm); log("knn2 warm-up"); ratio(warm); log("ratio warm-up")
    t_knn, t_ratio, st_knn, st_ratio, kept = [], [], None, None, 0
    for _ in range(args.reps):                                    # A B A B
        t0 = time.perf_counter(); r = knn2(pairs); t_knn.append(time.perf_counter() - t0); st_knn = m.stats()
        fb_knn = m.l2_last_fallback_rows()
        del r
        t0 = time.perf_counter(); r = ratio(pairs); t_ratio.append(time.perf_counter() - t0); st_ratio = m.stats()
        kept = int(r[4].sum())
        del r
        log(f"jobs {t_knn[-1]:.3f} / {t_ratio[-1]:.3f} s")
    spread = lambda t: (max(t) - min(t)) / min(t)
    frac = lambda t: evals * 2 * dim / t / BF16_PEAK
    line = {"workload": f"{n_img} images x {per} uniform [0,1) float descriptors, D {dim} (seed 5000 + image), "
                        f"{len(pairs)} pairs a < b, one GPU",
            "knn2_job": {"seconds": min(t_knn), "seconds_each": t_knn, "spread": spread(t_knn), "evals_per_s": evals / min(t_knn),
                         "frac_of_bf16_peak": frac(min(t_knn)), "fallback_rows": fb_knn, "stats": st_knn},
            "ratio_job": {"seconds": min(t_ratio), "seconds_each": t_ratio, "spread": spread(t_ratio),
                          "evals_per_s": evals / min(t_ratio), "frac_of_bf16_peak": frac(min(t_ratio)), "kept": kept,
                          "ratio": 0.8, "cross_check": True, "stats": st_ratio},
            "peak_note": "algorithmic: N1 N2 x 2 D flops per pair over the whole call's time, against the measured bf16 "
                         "1648.6 TFLOP/s of DESIGN.md section 4.2 (data sheet: 2250 dense)"}

    # the per-pair loop on a subset, alternated with the batch on the same subset
    sub = pairs[:min(args.subset, len(pairs))]
    lib, h = m._lib, m._h
    ob = [torch.empty(per, dtype=dt, device=dev) for dt in (torch.int32, torch.float32, torch.int32, torch.float32)]

    def loop():
        same = True
        with m.torch_ordered(dev):                        # the comparisons below run on torch's stream
            for p, (a, b) in enumerate(sub):
                m._check(lib.pgm_knn2_l2_dev(h, d_all[int(offs[a]):].data_ptr(), per, d_all[int(offs[b]):].data_ptr(), per,
                                             dim, *(o.data_ptr() for o in ob), None))
                if check is not None and p % 97 == 0:
                    same &= all(bool((o.view(torch.int32) == c[p * per:(p + 1) * per].view(torch.int32)).all())
                                for o, c in zip(ob, check))
        torch.cuda.synchronize()
        return same

    check = None
    knn2(sub); loop()
    t_loop, t_sub, same = [], [], True
    for _ in range(args.reps):
        t0 = time.perf_counter(); r = knn2(sub); t_sub.append(time.perf_counter() - t0)
        check = r[:4]
        t0 = time.perf_counter(); same &= loop(); t_loop.append(time.perf_counter() - t0)
    log("per-pair loop done")
    line["per_pair_loop"] = {"pairs": len(sub), "loop_seconds": min(t_loop), "batch_seconds": min(t_sub),
                             "loop_seconds_per_pair": min(t_loop) / len(sub), "batch_seconds_per_pair": min(t_sub) / len(sub),
                             "batch_speedup": min(t_loop) / min(t_sub), "sampled_pairs_bit_identical": bool(same),
                             "note": "pgm_knn2_l2_dev per pair (device buffers, no host copy), every 97th pair compared "
                                     "bit-exactly with the batch; alternated with the batch in the same process"}

    # the single-pair rate
    n = args.big
    g.manual_seed(77)
    q = torch.rand((n, dim), generator=g, device=dev); t = torch.rand((n, dim), generator=g, device=dev)
    out = [torch.empty(n, dtype=dt, device=dev) for dt in (torch.int32, torch.float32, torch.int32, torch.float32)]
    call = lambda: m._check(lib.pgm_knn2_l2_dev(h, q.data_ptr(), n, t.data_ptr(), n, dim, *(o.data_ptr() for o in out), None))
    call(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream(dev)
    m.set_stream(stream.cuda_stream)
    e0.record(stream)
    for _ in range(20):
        call()
    e1.record(stream); torch.cuda.synchronize()
    m.set_stream(None)
    ms = e0.elapsed_time(e1) / 20
    line["single_32768"] = {"n1": n, "n2": n, "dim": dim, "ms": ms, "evals_per_s": n * n / ms * 1e3,
                            "frac_of_bf16_peak": n * n * 2 * dim / (ms * 1e-3) / BF16_PEAK,
                            "timing": "CUDA events around 20 back-to-back calls"}
    del q, t, out
    log("single pair done")

    line["phases"] = {"knn2_job": phases(lambda: knn2(pairs)), "ratio_job": phases(lambda: ratio(pairs)),
                      "note": "torch.profiler in a separate pass; conversion = l2b_prep + l2b_split16, filter = "
                              "l2b_filter + l2b_scatter"}
    line["gpu"] = gpu_info()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    m.close()


main()
