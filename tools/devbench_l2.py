"""Developer bench for the float-L2 tcgen05 path."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from photogrammetry_b200.keypoint_matching import Matcher
m = Matcher(0); stream = torch.cuda.Stream(); m.set_stream(stream.cuda_stream)
peaks = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")) else {"bf16_tflops": 1648.6}
for n, dim in [(8192, 128), (32768, 128), (65536, 128), (32768, 64)]:
    with torch.cuda.stream(stream):
        q = torch.rand((n, dim), device="cuda"); t = torch.rand((n, dim), device="cuda")
        oj = torch.empty((2, n), dtype=torch.int32, device="cuda"); od = torch.empty((2, n), device="cuda")
    def run():
        m._check(m._lib.pgm_knn2_l2_dev(m._h, q.data_ptr(), n, t.data_ptr(), n, dim, oj[0].data_ptr(), od[0].data_ptr(), oj[1].data_ptr(), od[1].data_ptr(), None))
    for _ in range(3): run()
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(10): run()
    e1.record(stream); e1.synchronize()
    ms = e0.elapsed_time(e1) / 10
    dp = (dim + 63) // 64 * 64
    alg = 2.0 * dim * n * n / (ms * 1e-3) / 1e12
    print(json.dumps({"n": n, "dim": dim, "ms": ms, "evals_per_s": n * n / (ms * 1e-3), "algorithmic_tflops(2D per eval)": alg,
                      "algorithmic_frac_of_measured_bf16_peak": alg / peaks["bf16_tflops"],
                      "executed_frac": 2.0 * dp * n * n / (ms * 1e-3) / 1e12 / peaks["bf16_tflops"],
                      "fallback_rows": m.l2_last_fallback_rows()}))
