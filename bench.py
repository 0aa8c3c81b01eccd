#!/usr/bin/env python
"""bench.py -- headline benchmark of the descriptor-matching hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[4], the configuration the metric "... at 1/2/4/8 B200" is quoted on): synthetic
all-pairs matching of 512 images x 4096 256-bit descriptors = 130 816 image pairs = 2.195e12 distance evaluations,
every pair matched with the reference's semantics (full Hamming matrix + greedy one-to-one assignment,
KeypointMatching.cs:14-69; the caller is TestService.cs:80-96 generalised to many pairs).  One step = the whole
job.  At N > 1 the pair list is cut into N contiguous cost-balanced blocks (sharding.partition_pairs), one per
rank; image pairs are independent units, so there is NO data-path collective (strong scaling of a fixed job).

metric  = distance evaluations per second: N1*N2 per pair (each (i,j) counted once, however many passes
          recompute it), whole job over all ranks / max-over-ranks device time.
value   = descriptors and triples resident in HBM (pgm_match_pairs_batch_dev), CUDA events on the launching stream.
e2e     = the same through the host-buffer C-ABI call (pgm_match_pairs_batch): page-locked host descriptors in,
          page-locked host triples out, H2D + D2H inside the timed region, wall clock.
roofline= integer pipe: one 256-bit distance = 8 POPC.32 (SURVEY 8d); the denominator is a POPC micro-benchmark
          run live on the same GPU (MEASURED_PEAKS.json has no integer-pipe figure).
cpu_baseline / --impl reference = the oracle's literal restatement of the C# algorithm (kind "port": the C#
          itself cannot run here, no dotnet).
extras  = configs[1] (one 8192 x 8192 pair, latency), configs[2] proxy (K=32 shifted-star sequence), configs[3]
          (200k x 200k, train-sharded over the ranks), nearest/second-nearest and float-L2 passes.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "descriptor distance-evals/s (greedy MatchKeypoints, 256-bit Hamming, all-pairs)"
UNIT = "evals/s"
BITS, STRIDE = 256, 32


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--images", type=int, default=512, help="images of the all-pairs job")
    ap.add_argument("--per", type=int, default=4096, help="descriptors per image")
    ap.add_argument("--cpu-sample", type=int, default=2048, help="rows/cols of the per-step CPU sample of one pair")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[1]/[2]/[3], knn and float-L2 extras")
    ap.add_argument("--no-full-unit", action="store_true", help="reference arm: skip the one full-size 4096x4096 pair")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def workload_name(args, world):
    n_pairs = args.images * (args.images - 1) // 2
    return (f"configs[4]: synthetic all-pairs matching, {args.images} images x {args.per} descriptors "
            f"({n_pairs} pairs, {n_pairs * args.per * args.per:.4g} distance evals), 256-bit, uniform per image "
            f"(seed = 9000 + image index)")


def make_images(args):
    from photogrammetry_b200 import synthetic
    imgs = np.concatenate([synthetic.uniform_descriptors(9000 + k, args.per, BITS) for k in range(args.images)])
    offs = np.arange(args.images + 1, dtype=np.int64) * args.per
    return imgs, offs


# --------------------------------------------------------------------------
# clocks (recipe: /opt/skills/guides/B200_PROFILING.md)
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        hi = [x for x in sm if x >= 0.5 * max(sm)]          # "under load": the upper half of the observed range
        return {"sm_mhz": float(np.median(hi)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------
# CPU side (the oracle: test infrastructure, used here only as the timed baseline)
# --------------------------------------------------------------------------
def cpu_literal_parallel(pairs_qt, threads: int) -> float:
    """Run the literal restatement (1 thread per pair, like the single-threaded C#) on `threads` pairs at once --
    image pairs are independent, so that is how a host would use all its cores.  Returns wall seconds."""
    from oracle import orc
    err = []

    def work(k):
        try:
            orc.match_literal(pairs_qt[k][0], pairs_qt[k][1], kernighan=True)
        except Exception as e:  # pragma: no cover
            err.append(e)
    ths = [threading.Thread(target=work, args=(k,)) for k in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    if err:
        raise err[0]
    return dt


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def run_reference(args, rank: int):
    """The reference's own CPU algorithm (oracle port of KeypointMatching.cs:14-82) on the box's host cores: every
    thread matches one image pair of the job (single-threaded per pair, like the C#).  A step is a bounded sample --
    the leading cpu_sample x cpu_sample block of `threads` pairs of the job; one full-size 4096 x 4096 pair per
    thread is timed once so the line can state what the sample's rate overstates (the scan phase is cubic)."""
    if rank != 0:
        return
    imgs, offs = make_images(args)
    T = host_threads()
    s = min(args.cpu_sample, args.per)

    def pair(k, size):
        a, b = k % args.images, (k + 1 + k // args.images) % args.images
        return imgs[offs[a]:offs[a] + size], imgs[offs[b]:offs[b] + size]
    sample_pairs = [pair(k, s) for k in range(T)]
    for _ in range(min(args.warmup, 1)):
        cpu_literal_parallel(sample_pairs, T)
    times = [cpu_literal_parallel(sample_pairs, T) for _ in range(args.steps)]
    Tt = float(np.sum(times))
    value = T * float(s) * s * args.steps / Tt
    full = None
    if not args.no_full_unit and s < args.per:
        dt = cpu_literal_parallel([pair(k, args.per) for k in range(T)], T)
        full_rate = T * float(args.per) * args.per / dt
        full = {"pairs": T, "size": args.per, "seconds": dt, "value": full_rate, "unit": UNIT,
                "sample_to_full_size_factor": full_rate / value,
                "note": "full-size units of the job (one 4096x4096 pair per thread), timed once; the per-step sample "
                        "overstates the reference's rate by 1/factor because the argmin scans are cubic"}
    sample = (f"{T} pairs at once (1 thread each, like the single-threaded C#), leading {s}x{s} block of each "
              f"{args.per}x{args.per} pair; literal O(N^3) restatement of KeypointMatching.cs:14-82 (Kernighan CountOnes, "
              f"full matrix, N1 argmin scans)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * Tt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32 (XOR + popcount)", "data": "synthetic",
        "config": {"workload": workload_name(args, 1), "cpu_sample": s, "threads": T},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": T, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if full:
        line["full_size_unit"] = full
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------
def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist

    from photogrammetry_b200 import sharding
    from photogrammetry_b200._lib import pinned_empty
    from photogrammetry_b200.keypoint_matching import Matcher

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    per = args.per

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    imgs, offs = make_images(args)
    pairs = sharding.all_pairs(args.images)
    lo, hi = sharding.shard_for_rank(pairs, np.diff(offs), rank, world)
    mine = np.ascontiguousarray(pairs[lo:hi])
    rows = len(mine) * per
    total_evals = float(len(pairs)) * per * per

    m = Matcher(local_rank)
    stream = torch.cuda.Stream(device=dev)
    m.set_stream(stream.cuda_stream)
    with torch.cuda.stream(stream):
        d_all = torch.from_numpy(imgs).to(dev)
        d_out = torch.empty((3, max(rows, 1)), dtype=torch.int32, device=dev)
    stream.synchronize()

    def step_dev():
        return m.match_pairs_batch_dev(d_all.data_ptr(), offs, mine, BITS, STRIDE, d_out[0].data_ptr(),
                                       d_out[1].data_ptr(), d_out[2].data_ptr(), rows)

    # ---- value: device-resident, CUDA events on the launching stream.  The job's working set (64 MB of descriptors,
    # >1 GB of matcher state per chunk of 4096 pairs, 6.4 GB / N of triples) is far larger than the 126 MB L2.
    for _ in range(max(args.warmup, 3)):
        step_dev()
    stream.synchronize()
    st_dev = m.stats()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    with torch.cuda.stream(stream):
        for k in range(args.steps):
            ev[k][0].record(stream)
            counts = step_dev()
            ev[k][1].record(stream)
    stream.synchronize()
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_out, counts, len(pairs), lo, hi, per, rank, world, dev)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    T_ms = max_over_ranks(float(np.sum(step_ms)))
    value = total_evals * args.steps / (T_ms * 1e-3)
    launches = sum_over_ranks(float(st_dev["kernel_launches"])) * args.steps

    # ---- e2e: host buffers through the C ABI, wall clock, H2D + D2H inside.  Inputs and outputs live in page-locked
    # host memory (pgm_host_alloc), which the library copies from / to directly, chunk k's triples leaving while
    # chunk k + 1 computes.
    p_imgs = pinned_empty(imgs.shape, np.uint8)
    p_imgs[:] = imgs
    p_out = pinned_empty((3, max(rows, 1)), np.int32)
    p_out[:] = 0
    e2e_steps = max(2, args.steps // 5)
    m.match_pairs_batch(p_imgs, offs, mine, BITS, out=p_out)       # (also sizes the library's double buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        soa, _starts, _counts = m.match_pairs_batch(p_imgs, offs, mine, BITS, out=p_out)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    st_host = m.stats()
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = total_evals * e2e_steps / e2e_s
    h2d = sum_over_ranks(float(st_host["h2d_bytes"]))
    d2h = sum_over_ranks(float(st_host["d2h_bytes"]))
    # the two paths agree on this rank's first and last pair
    chk = d_out[:, :per].cpu().numpy()
    assert (chk == soa[:, :per]).all() and (d_out[:, rows - per:rows].cpu().numpy() == soa[:, rows - per:rows]).all()

    # ---- roofline of the dominant kernel: the round-0 launch of hamming_round_kernel<8> (all N1 x N2 distances of
    # every pair of a chunk + row / column argmin + candidate edges); profiled on this rank's first chunk.
    popc_peak, lop3_peak = m.measure_popc_peak(300)
    chunk_pairs = mine[:min(len(mine), 2048)]            # (one chunk of the batch engine: <= 24 M row + column slots)
    m.set_profiling(True)
    prof = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        m.match_pairs_batch_dev(d_all.data_ptr(), offs, chunk_pairs, BITS, STRIDE, d_out[0].data_ptr(),
                                d_out[1].data_ptr(), d_out[2].data_ptr(), rows)
        e1.record(stream)
        e1.synchronize()
        ms, evals = m.round_profile()
        prof.append((e0.elapsed_time(e1), ms, evals, m.stats()))
    m.set_profiling(False)
    chunk_ms, pm, pe, st_chunk = prof[-1]
    chunk_evals = float(len(chunk_pairs)) * per * per
    r0_ms, r0_evals = float(pm[0]), float(pe[0])
    achieved = r0_evals * 8 / (r0_ms * 1e-3)                          # POPC.32-equivalents / s, round-0 launch
    per_gpu_value = value / world
    roofline = {
        "bound": "int-pipe",
        "bound_note": "POPC.32 issue rate (SURVEY 8d); neither HBM nor the tensor pipe bounds this path",
        "kernel": "hamming_round_kernel<8>, round-0 launch of a chunk of pairs (every N1 x N2 distance once + row/column "
                  "argmin + candidate edges)",
        "achieved": achieved / 1e9, "peak": popc_peak / 1e9, "unit": "Gpopc32/s", "frac": achieved / popc_peak,
        "peak_source": "measured live: register-only POPC micro-benchmark on this GPU (pgm_measure_popc_peak); "
                       "nominal 148 SM x 16/clk x 1.965 GHz = 4654",
        "algorithmic": "8 POPC.32 per 256-bit distance (SURVEY 8d) x the N1*N2 distances of the launch's pairs",
        "note": "the kernel uses a carry-save popcount (5 POPC + 14 LOP3 per distance), which is how frac can exceed "
                "1.0 of the plain 8-POPC roofline; frac_vs_carry_save_bound is the same launch against 5 POPC per distance",
        "frac_vs_carry_save_bound": achieved * 5.0 / 8.0 / popc_peak,
        "whole_call_frac": per_gpu_value * 8 / popc_peak,
        "whole_call_note": "value (whole job, every pass, accept / sparse / finisher / ordering kernels, host planning "
                           "syncs) per GPU x 8 POPC per distance / peak",
        "lop3_peak_gops": lop3_peak / 1e9,
        "launch_ms": r0_ms, "launches_per_chunk": int(len(pm)),
        "kernel_share_of_step": float(r0_ms / chunk_ms),
        "all_round_launches_share_of_step": float(np.sum(pm) / chunk_ms),
        "profiled_chunk": {"pairs": int(len(chunk_pairs)), "ms": chunk_ms, "evals": chunk_evals,
                           "recompute_factor": st_chunk["evals_computed"] / max(1, st_chunk["distance_evals"]),
                           "distance_passes": st_chunk["rounds"]},
        "hbm_gbs_for_context": float((imgs.nbytes + 12.0 * rows) / (np.mean(step_ms) * 1e-3) / 1e9),
        "traffic": None,
        "traffic_note": "not an HBM-bound kernel; dram bytes of the launch are in profiles/r02_ncu_round_kernel.json",
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": T_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 (XOR + popcount)", "data": "synthetic",
        "config": {"workload": workload_name(args, world), "images": args.images, "descriptors_per_image": per,
                   "pairs": int(len(pairs)), "desc_bits": BITS,
                   "l2": "inputs larger than L2: 64 MB of descriptors, > 1 GB of matcher state per chunk of 4096 pairs and "
                         "6.4 GB / N of triples stream through the 126 MB L2 every step (no flush needed)",
                   "parallelism": f"pair-sharded x{world} (contiguous cost-balanced blocks of the pair list), no collective"},
        "matched_pairs_per_s": float(len(pairs)) * per * args.steps / (T_ms * 1e-3),
        "distance_passes_per_chunk": st_dev["rounds"] / max(1, (len(mine) + 4095) // 4096),
        "recompute_factor": st_dev["evals_computed"] / max(1, st_dev["distance_evals"]),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                "host_memory": "page-locked descriptors and result arrays (pgm_host_alloc); H2D of all descriptors and D2H "
                               "of every triple inside the timed region, per rank"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "clocks": clocks,
    }
    del p_out, p_imgs, d_out

    if not args.no_extras:
        ex = {}
        try:
            ex.update(extra_sharded_pair(m, stream, dev, rank, world, popc_peak))       # all ranks: has collectives
        except Exception as e:  # pragma: no cover
            ex["configs3_200k_train_sharded"] = {"error": repr(e)}
        if rank == 0:
            for fn in (extra_single_pair, extra_sequence, extra_knn_l2):
                try:
                    ex.update(fn(m, stream, dev, popc_peak))
                except Exception as e:  # pragma: no cover
                    ex[fn.__name__] = {"error": repr(e)}
        line["extras"] = ex

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import orc
        a, b = imgs[offs[0]:offs[1]], imgs[offs[1]:offs[2]]
        t0 = time.perf_counter()
        orc.match_literal(a, b, kernighan=True)
        secs = time.perf_counter() - t0
        line["cpu_baseline"] = {
            "value": per * float(per) / secs, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"1 of the job's {len(pairs)} pairs at full size ({per}x{per}): oracle literal restatement of "
                      f"KeypointMatching.cs:14-82 (Kernighan CountOnes, full matrix, cubic argmin scans), 1 thread like "
                      f"the C#, {secs:.1f} s"}
        try:
            t0 = time.perf_counter()
            for k in range(4):
                orc.match_sweep(imgs[offs[k]:offs[k + 1]], imgs[offs[k + 1]:offs[k + 2]])
            dt = time.perf_counter() - t0
            line["cpu_fast"] = {"value": 4 * per * float(per) / dt, "unit": UNIT, "cores": orc.num_threads(),
                                "what": "oracle counting-sort sweep (popcnt, OpenMP) on 4 full pairs of the job, same output"}
        except Exception as e:  # pragma: no cover
            line["cpu_fast"] = {"error": str(e)}
    m.close()
    if rank == 0:
        print(json.dumps(line), flush=True)


DUMP_BYTES = 64_000_000        # --dump-outputs writes at most this much (64 MB)


def dump_outputs(out_dir, d_out, counts, n_pairs, lo, hi, per, rank, world, dev):
    """--dump-outputs: what the timed call returned to its caller in the last timed step, as float64 arrays (exact for
    every int32), so that two builds can be compared output for output on the same seeded job.

        counts.npy       [n_pairs]   triples written for each pair of the job (the counts the call returns)
        pair_index.npy   [S]         a fixed sample of the job's pairs (seed 0, ascending): as many as fit DUMP_BYTES
        query_index.npy  [S, per]    the sampled pairs' triples (query index, train index, Hamming distance) in the
        train_index.npy  [S, per]    order the call wrote them
        distance.npy     [S, per]

    Every rank contributes the pairs of its block [lo, hi) of the pair list; rank 0 writes the files."""
    import torch
    import torch.distributed as dist

    room = DUMP_BYTES - 5 * 256 - 8 * n_pairs                   # five .npy headers and counts.npy
    n_sample = min(n_pairs, max(0, room // (8 + 3 * 8 * per)))
    sample = np.sort(np.random.default_rng(0).choice(n_pairs, n_sample, replace=False))
    owned = np.flatnonzero((sample >= lo) & (sample < hi))
    tri = torch.zeros((3, n_sample, per), dtype=torch.int32, device=dev)
    cnt = torch.zeros(n_pairs, dtype=torch.int32, device=dev)
    if len(owned):
        # every image has `per` descriptors, so pair p of the block owns rows (p - lo) * per ... + per
        rows = torch.from_numpy((sample[owned] - lo) * per).to(dev)[:, None] + torch.arange(per, device=dev)[None, :]
        tri[:, torch.from_numpy(owned).to(dev)] = d_out[:, rows]
    cnt[lo:hi] = torch.from_numpy(np.ascontiguousarray(counts, dtype=np.int32)).to(dev)
    if world > 1:
        dist.all_reduce(tri)
        dist.all_reduce(cnt)
    if rank != 0:
        return
    tri, cnt = tri.cpu().numpy(), cnt.cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"counts": cnt, "pair_index": sample, "query_index": tri[0], "train_index": tri[1], "distance": tri[2]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


# --------------------------------------------------------------------------
# extras
# --------------------------------------------------------------------------
def _time_stream(fn, stream, warm=3, reps=10):
    import torch
    for _ in range(warm):
        fn()
    stream.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def extra_single_pair(m, stream, dev, popc_peak):
    """configs[1]: one 8192 x 8192 pair (latency mode: init + round 0 + one persistent kernel), device resident and
    through host buffers."""
    import torch

    from photogrammetry_b200 import synthetic
    from photogrammetry_b200._lib import pinned_empty
    out = {}
    n = 8192
    for dist_name in ("U", "C"):
        q, t = synthetic.config2_pair(n, dist_name)
        with torch.cuda.stream(stream):
            d_q, d_t = torch.from_numpy(q).to(dev), torch.from_numpy(t).to(dev)
            o = torch.empty((3, n), dtype=torch.int32, device=dev)
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        stream.synchronize()

        def step():
            m.match_greedy_dev(d_q.data_ptr(), n, d_t.data_ptr(), n, BITS, STRIDE, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), n)
        for _ in range(3):
            step()
        ts = []
        with torch.cuda.stream(stream):
            for k in range(20):
                flush.fill_(k & 0xFF)                                   # L2 flush between timed calls
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream); step(); e1.record(stream)
                ts.append((e0, e1))
        stream.synchronize()
        ms = float(np.median([a.elapsed_time(b) for a, b in ts]))
        st = m.stats()
        tb = []
        with torch.cuda.stream(stream):                                 # the same call back to back (state and code stay in L2)
            for k in range(20):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream); step(); e1.record(stream)
                tb.append((e0, e1))
        stream.synchronize()
        ms_b2b = float(np.median([a.elapsed_time(b) for a, b in tb]))
        rec = {"ms": ms, "evals_per_s": n * n / (ms * 1e-3), "whole_call_frac_of_popc_peak": n * n * 8 / (ms * 1e-3) / popc_peak,
               "ms_back_to_back": ms_b2b, "whole_call_frac_back_to_back": n * n * 8 / (ms_b2b * 1e-3) / popc_peak,
               "distance_passes": st["rounds"], "recompute_factor": st["evals_computed"] / st["distance_evals"],
               "launches": st["kernel_launches"], "l2": "ms: flushed between timed calls; ms_back_to_back: not flushed"}
        if dist_name == "U":
            m.set_profiling(True)
            r0 = []
            for _ in range(4):
                step()
                a, _b = m.round_profile()
                r0.append(float(a[0]))
            m.set_profiling(False)
            rec["round0_launch_ms"] = float(np.median(r0[1:]))
            rec["round0_frac_of_popc_peak"] = n * n * 8 / (rec["round0_launch_ms"] * 1e-3) / popc_peak
            rec["dominant"] = ("tail_kernel<8> (every pass after round 0: accept, candidate-edge filter, sparse sub-rounds, "
                               "finisher, ordering) when its share exceeds round 0's")
            rec["tail_share_of_call"] = 1.0 - rec["round0_launch_ms"] / ms
            pq, pt, po = pinned_empty(q.shape, np.uint8), pinned_empty(t.shape, np.uint8), pinned_empty((3, n), np.int32)
            pq[:] = q; pt[:] = t
            for _ in range(3):
                m.match_greedy(pq, pt, BITS, out=po)
            t0 = time.perf_counter()
            for _ in range(20):
                m.match_greedy(pq, pt, BITS, out=po)
            rec["e2e_host_buffers_ms"] = (time.perf_counter() - t0) / 20 * 1e3
        out[f"configs1_pair_8192_{dist_name}"] = rec
        del d_q, d_t, o, flush
    return out


def extra_sequence(m, stream, dev, popc_peak):
    """configs[2] proxy (SURVEY D5): K = 32 frames of the 15-point star shifted right by 5 k px, FAST + BRIEF on the
    device, consecutive frames matched greedily and with ratio 0.8 + cross-check."""
    from photogrammetry_b200 import sequence
    return {"configs2_star_sequence_K32": sequence.bench_star_sequence(m, stream, dev)}


def extra_knn_l2(m, stream, dev, popc_peak):
    import torch

    from photogrammetry_b200 import synthetic
    out = {}
    n = 8192
    q, t = synthetic.config2_pair(n, "U")
    with torch.cuda.stream(stream):
        d_q, d_t = torch.from_numpy(q).to(dev), torch.from_numpy(t).to(dev)
        o = torch.empty((4, n), dtype=torch.int32, device=dev)
    stream.synchronize()
    lib, h = m._lib, m._h

    def knn():
        lib.pgm_knn2_hamming_dev(h, d_q.data_ptr(), n, d_t.data_ptr(), n, BITS, STRIDE, *(o[k].data_ptr() for k in range(4)))
    ms, _ = _time_stream(knn, stream, reps=20)
    out["knn2_8k"] = {"ms": ms, "evals_per_s": n * n / (ms * 1e-3), "frac_of_popc_peak": n * n * 8 / (ms * 1e-3) / popc_peak}

    # float descriptors (north_star extension): squared-L2 top-2 on tcgen05, whole call (operand split, GEMM with the
    # norms folded in, exact refinement), device resident; roofline = tensor pipe, measured bf16 peak
    peak_tf, peak_src = 1590.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"
    try:
        peak_tf = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
        peak_src = "MEASURED_PEAKS.json bf16_tflops (burst)"
    except Exception:
        pass
    for nf in (8192, 32768):
        dim = 128
        g = torch.Generator(device=dev); g.manual_seed(7)
        with torch.cuda.stream(stream):
            fq = torch.rand((nf, dim), device=dev, generator=g)
            ft = torch.rand((nf, dim), device=dev, generator=g)
            fj = torch.empty((2, nf), dtype=torch.int32, device=dev)
            fd = torch.empty((2, nf), device=dev)
        stream.synchronize()

        def l2():
            m._check(lib.pgm_knn2_l2_dev(h, fq.data_ptr(), nf, ft.data_ptr(), nf, dim, fj[0].data_ptr(), fd[0].data_ptr(),
                                         fj[1].data_ptr(), fd[1].data_ptr(), None))
        ms, _ = _time_stream(l2, stream, reps=10)
        # observed index mismatch rate against an exact fp32 search (torch, fp32 cdist on a row sample)
        with torch.cuda.stream(stream):
            rows = torch.arange(0, nf, max(1, nf // 2048), device=dev)[:2048]
            dd = (fq[rows] * fq[rows]).sum(1, keepdim=True) - 2.0 * fq[rows].double() @ ft.double().T + (ft.double() * ft.double()).sum(1)[None, :]
            ref_j = dd.argmin(1).to(torch.int32)
            mism = float((ref_j != fj[0][rows]).float().mean().item())
            ref_d = dd.gather(1, fj[0][rows].long()[:, None])[:, 0]
            rel = float(((fd[0][rows].double() - ref_d).abs() / ref_d.clamp_min(1e-30)).max().item())
        stream.synchronize()
        tf_alg = 2.0 * dim * nf * nf / (ms * 1e-3) / 1e12
        st = m.stats()
        fallback_rows = m.l2_last_fallback_rows()
        fp16 = fallback_rows >= 0
        terms = 1.0 if fp16 else 3.0
        out[f"l2_knn2_{nf // 1024}k_d{dim}"] = {
            "ms": ms, "evals_per_s": nf * float(nf) / (ms * 1e-3), "launches": st["kernel_launches"],
            "ranking": ("one fp16 term under a global power-of-two scale, certified band, exhaustive fallback for "
                        "uncertified rows" if fp16 else "three-term bf16 split (PGM_L2_MODE=bf16x3)"),
            "rows_recomputed_exhaustively": fallback_rows,
            "nearest_index_mismatch_rate_vs_fp64": mism, "nearest_distance_max_rel_err_vs_fp64": rel,
            "roofline": {"bound": "tensor", "achieved": tf_alg, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf_alg / peak_tf,
                         "peak_source": peak_src,
                         "algorithmic": "2 x D flops per distance (SURVEY 8d)",
                         "executed_frac": terms * (dim + 16.0) / dim * tf_alg / peak_tf if fp16 else terms * tf_alg / peak_tf,
                         "executed": ("2 x (D + 16) per distance: one fp16 GEMM pass + the K = 16 norm step; the kernel is "
                                      "bound by the epilogue's TMEM reads and the operand feed, not by the tensor pipe "
                                      "(DESIGN 4.2)" if fp16 else
                                      "2 x 3 x D per distance: three bf16 split terms (hi.hi + lo.hi + hi.lo); the norm "
                                      "MMA adds 4 %")}}
        del fq, ft, fj, fd
    return out


def extra_sharded_pair(m, stream, dev, rank, world, popc_peak):
    """configs[3]: one 200k x 200k pair, train set sharded over the ranks (pgm_multi: NCCL inside the library)."""
    from photogrammetry_b200 import sharding
    return {"configs3_200k_train_sharded": sharding.bench_train_sharded(m, stream, dev, rank, world, popc_peak)}


def main():
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
