#!/usr/bin/env python
"""Ratio test + cross-check of every pair of an image set (pgm_match_ratio_crosscheck_pairs_batch_dev), BASELINE configs[4].

    python tools/bench_ratio_allpairs.py [--images 512 --per 4096]                 # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port P \
        tools/bench_ratio_allpairs.py                                             # G GPUs

As tools/bench_allpairs.py: every rank holds all descriptors and takes a contiguous, cost-balanced block of the pair list
(sharding.shard_for_rank); there is no collective but the timing barrier and max-reduce.  One JSON line (rank 0):
  ratio_job      the whole job, device resident, ratio 0.8 + cross-check: seconds, distances/s, share of the live-measured
                 POPC peak (8 POPC per 256-bit distance)
  greedy_job     the greedy matcher (pgm_match_pairs_batch_dev) on the same job, alternated with the ratio job (A B A B)
  per_pair_route pgm_match_ratio_crosscheck (host buffers, one pair per call) on sampled pairs, extrapolated to the job
  pair_65536     one 65 536 x 65 536 pair: call time and the kernel split (torch.profiler, its own run)
  configs2_sequence  the 31 consecutive pairs of the configs[2] star sequence: this entry point vs the one-CTA batch
  gpu            name, power limit and max SM clock (read-only nvidia-smi query in the same run)
and checks that the sampled pairs are bit-identical to the per-pair entry point."""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from photogrammetry_b200 import sequence, sharding, synthetic
from photogrammetry_b200.keypoint_matching import Matcher

RATIO, CROSS = 0.8, True


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return [dict(zip(("name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(",")))) for line in out]
    except Exception as e:  # pragma: no cover
        return [{"error": str(e)}]


def kernel_split(m, d_all, offs, pairs):
    """Device time per kernel of one call (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, pairs, 256, RATIO, CROSS, -1)
        torch.cuda.synchronize()
    split = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        for key in ("knn2_cols_pairs_kernel", "rcp_filter_kernel", "rcp_scatter_kernel"):
            if key in e.key:
                split[key] = split.get(key, 0.0) + us * 1e-3
    return split


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--per", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3, help="A B pairs of the ratio job and the greedy job")
    ap.add_argument("--sample", type=int, default=512, help="pairs timed through the per-pair entry point")
    ap.add_argument("--big", type=int, default=65536)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local); dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_img, per = args.images, args.per
    imgs = np.concatenate([synthetic.uniform_descriptors(9000 + k, per, 256) for k in range(n_img)])
    offs = np.arange(n_img + 1, dtype=np.int64) * per
    pairs = sharding.all_pairs(n_img)
    lo, hi = sharding.shard_for_rank(pairs, np.diff(offs), rank, world)
    mine = pairs[lo:hi]
    m = Matcher(local)
    stream = torch.cuda.Stream(device=dev); torch.cuda.set_stream(stream); m.set_stream(stream.cuda_stream)
    d_all = torch.from_numpy(imgs).to(dev)
    d_o = torch.empty((3, len(mine) * per), dtype=torch.int32, device=dev)

    def sync_all():
        if world > 1: dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):
        if world == 1: return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX); return float(tt.item())

    def run_ratio():
        r = m.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, mine, 256, RATIO, CROSS, -1)
        torch.cuda.synchronize()
        return r

    def run_greedy():
        m.match_pairs_batch_dev(d_all.data_ptr(), offs, mine, 256, 32, d_o[0].data_ptr(), d_o[1].data_ptr(),
                                d_o[2].data_ptr(), len(mine) * per)
        torch.cuda.synchronize()

    popc_peak, _ = m.measure_popc_peak(300)
    warm = mine[:min(len(mine), 256)]
    m.match_ratio_crosscheck_pairs_batch_dev(d_all, offs, warm, 256, RATIO, CROSS, -1)
    m.match_pairs_batch_dev(d_all.data_ptr(), offs, warm, 256, 32, d_o[0].data_ptr(), d_o[1].data_ptr(), d_o[2].data_ptr(),
                            len(mine) * per)
    torch.cuda.synchronize()
    t_ratio, t_greedy, res, st_ratio = [], [], None, None
    for _ in range(args.reps):                                     # A B A B
        sync_all(); t0 = time.perf_counter(); res = run_ratio(); t_ratio.append(maxr(time.perf_counter() - t0))
        st_ratio = m.stats()
        sync_all(); t0 = time.perf_counter(); run_greedy(); t_greedy.append(maxr(time.perf_counter() - t0))
    evals = float(len(pairs)) * per * per
    out, starts, counts = res
    spread = lambda t: (max(t) - min(t)) / min(t)
    line = {"workload": f"configs[4] ratio test + cross-check: {n_img} images x {per} uniform 256-bit descriptors "
                        f"(seed 9000 + image), {len(pairs)} pairs, ratio {RATIO}, cross-check, pair-sharded x{world}",
            "n_gpus": world, "pairs_total": int(len(pairs)), "pairs_rank0": int(len(mine)),
            "popc_peak_gpopc_s": popc_peak / 1e9,
            "ratio_job": {"seconds": min(t_ratio), "seconds_each": t_ratio, "spread": spread(t_ratio),
                          "evals_per_s": evals / min(t_ratio),
                          "frac_of_popc_peak_per_gpu": evals / world * 8 / min(t_ratio) / popc_peak,
                          "kept_rank0": int(counts.sum()), "rank0_stats": st_ratio},
            "greedy_job": {"seconds": min(t_greedy), "seconds_each": t_greedy, "spread": spread(t_greedy),
                           "evals_per_s": evals / min(t_greedy),
                           "frac_of_popc_peak_per_gpu": evals / world * 8 / min(t_greedy) / popc_peak},
            "ratio_over_greedy_time": min(t_ratio) / min(t_greedy),
            "peak_note": "share of peak = N1*N2 distances x 8 POPC.32 (plain 256-bit popcount) per GPU over the time of "
                         "the whole call, against pgm_measure_popc_peak measured in the same run"}
    if rank == 0:
        # the per-pair route on sampled pairs; also the bit-exactness check of those pairs
        idx = np.linspace(0, len(mine) - 1, min(args.sample, len(mine))).astype(int)
        host_out = out.cpu().numpy()
        same = True
        t_pp = 0.0
        for p in idx:
            a, b = mine[p]
            q, t = imgs[offs[a]:offs[a + 1]], imgs[offs[b]:offs[b + 1]]
            t0 = time.perf_counter()
            one = m.match_ratio_crosscheck(q, t, RATIO, CROSS, -1, 256)
            t_pp += time.perf_counter() - t0
            same &= bool((host_out[:, starts[p]:starts[p] + counts[p]].T == one).all())
        per_call = t_pp / len(idx)
        line["per_pair_route"] = {"sampled_pairs": int(len(idx)), "seconds_per_pair": per_call,
                                  "extrapolated_job_seconds_1gpu": per_call * len(pairs),
                                  "note": "pgm_match_ratio_crosscheck, host buffers, one pair per call (two distance "
                                          "passes, H2D + one synchronisation per call); job time EXTRAPOLATED from "
                                          "the sample, not measured"}
        line["sampled_pairs_bit_identical_to_per_pair_call"] = same

        # one big pair: call time, then the kernel split in a profiled call of its own
        n = args.big
        q = synthetic.uniform_descriptors(77, n, 256)
        t = synthetic.noisy_copy_descriptors(78, q, 256)
        d_big = torch.from_numpy(np.concatenate([q, t])).to(dev)
        boffs = np.array([0, n, 2 * n], dtype=np.int64)
        m.match_ratio_crosscheck_pairs_batch_dev(d_big, boffs, [(0, 1)], 256, RATIO, CROSS, -1)
        ts = []
        for _ in range(5):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            bo, bs, bc = m.match_ratio_crosscheck_pairs_batch_dev(d_big, boffs, [(0, 1)], 256, RATIO, CROSS, -1)
            ts.append(time.perf_counter() - t0)
        bst = m.stats()
        split = kernel_split(m, d_big, boffs, [(0, 1)])
        tot = sum(split.values())
        line["pair_65536"] = {"n1": n, "n2": n, "call_ms": min(ts) * 1e3, "evals_per_s": n * n / min(ts),
                              "frac_of_popc_peak": n * n * 8 / min(ts) / popc_peak, "kept": int(bc[0]),
                              "kernel_ms": split,
                              "filter_and_compaction_share_of_kernel_time":
                                  (tot - split.get("knn2_cols_pairs_kernel", 0.0)) / tot if tot else None,
                              "stats": bst}
        one = m.match_ratio_crosscheck(q, t, RATIO, CROSS, -1, 256)
        line["pair_65536"]["bit_identical_to_per_pair_call"] = bool((bo[:, :bc[0]].T.cpu().numpy() == one).all())
        del d_big

        # configs[2]: the star sequence's consecutive pairs, this entry point vs the one-CTA-per-pair batch
        frames = sequence.shifted_frames(sequence.star_gray(), 32, 5).astype(np.float32)
        d_frames = torch.from_numpy(frames).to(dev)
        xy, _sc, desc, kcounts = m.detect_describe_batch_dev(d_frames, 50.0, sequence.pairs_table(sequence.star_pairs()),
                                                             capacity=4096, python_generation=True)
        soffs = np.concatenate([[0], np.cumsum(kcounts)]).astype(np.int64)
        d_desc = torch.cat([desc[f, :int(kcounts[f])] for f in range(len(kcounts))]).contiguous()
        plist = sharding.consecutive_pairs(len(kcounts))
        calls = {"pairs_batch": m.match_ratio_crosscheck_pairs_batch_dev, "one_cta_batch": m.match_ratio_crosscheck_batch_dev}
        outs, times = {}, {k: [] for k in calls}
        for k, f in calls.items():
            outs[k] = f(d_desc, soffs, plist, 256, RATIO, CROSS, -1)
        for _ in range(50):
            for k, f in calls.items():
                torch.cuda.synchronize(); t0 = time.perf_counter()
                f(d_desc, soffs, plist, 256, RATIO, CROSS, -1)
                times[k].append(time.perf_counter() - t0)
        (ao, as_, ac), (bo2, bs2, bc2) = outs["pairs_batch"], outs["one_cta_batch"]
        eq = bool((ac == bc2).all()) and all(
            bool((ao[:, as_[p]:as_[p] + ac[p]] == bo2[:, bs2[p]:bs2[p] + bc2[p]]).all()) for p in range(len(plist)))
        line["configs2_sequence"] = {"pairs": int(len(plist)), "keypoints": int(soffs[-1]),
                                     "ms_pairs_batch": float(np.median(times["pairs_batch"])) * 1e3,
                                     "ms_one_cta_batch": float(np.median(times["one_cta_batch"])) * 1e3,
                                     "timing": "median of 50 alternated calls, each ending in its read-back of the counts",
                                     "identical_outputs": eq, "kept": int(ac.sum())}
        line["gpu"] = gpu_info()
        print(json.dumps(line), flush=True)
    m.close()
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


main()
