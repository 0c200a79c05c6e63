"""Measure pp.knn and pp.module.ICP (csrc/knn.cu) on one GPU and write profiles/knn_icp_bench.json.

    python tools/bench_knn.py [--reps 20] [--out profiles/knn_icp_bench.json]

Workloads (fp32, D = 3, uniform random clouds), on both sides of the N2 split rule (`splits` records which):
  * knn N1 = N2 = 1e5 with k = 1 and k = 16, and N1 = 2000, N2 = 1e5 with k = 8: too few queries to fill the GPU, so
    the N2 range is split over CTAs and a merge kernel follows;
  * knn N1 = 4e5, N2 = 1e5 with k = 1 and k = 16: enough queries, no split;
  * ICP on 8 x 1e5 points, 30 iterations (the stepper cannot stop earlier), no split.
Each time is taken with CUDA events around one call, repeated; median and min are reported.  Baselines in the same run:
a chunked torch.cdist + topk at the same sizes, and the reference's formula (norm of the broadcast difference, then
topk) at the largest size whose tensors stay within the memory budget below, next to pp.knn at that size.

The bound is the issue rate: each of the 4 schedulers of an SM issues at most one warp instruction per clock, so an SM
retires at most 128 thread instructions per clock, whatever pipe they use.  The instructions per distance evaluation are
counted in the SASS of the full-tile loop of knn_kernel<float, 3, 2, 1, false> (knn, k = 1) and of
knn_kernel<float, 3, 2, 1, true> (the ICP step): 169 instructions per trip of 4 points x 4 queries, i.e. 10.56 per
evaluation (3 FADD + 3 FFMA, then LOP3 key flip, ISETP + VIMNMX + SEL for the top-1 update, and the loads and loop
control shared by the trip).  For k > 1 the insertion into the top-k list is a data-dependent branch, so no single count
applies and no share is reported.  Memory is not the bound: the neighbour tiles are read from shared memory.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pypose_b200 as pp  # noqa: E402
from pypose_b200.function import _knn  # noqa: E402

REF_FORMULA_BYTES = 16 << 30      # budget for the reference formula's (N, N, 3) difference + (N, N) norm tensors
SASS_INSTR_PER_EVAL_K1 = 169 / 16 # see the module docstring


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True).stdout.strip().split(", ")
    props = torch.cuda.get_device_properties(0)
    return {"name": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2]),
            "sms": props.multi_processor_count}


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "reps": reps}


def cdist_topk(ref, nbr, k, chunk=8192):
    for i in range(0, ref.shape[0], chunk):
        torch.cdist(ref[i:i + chunk], nbr).topk(k, dim=-1, largest=False)


def reference_formula(ref, nbr, k):
    diff = ref.unsqueeze(-2) - nbr.unsqueeze(-3)
    return torch.linalg.norm(diff, dim=-1, ord=2).topk(k, dim=-1, largest=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "knn_icp_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_knn.py measures on a GPU"
    dev = torch.device("cuda:0")
    info = gpu_info()
    bound = info["sms"] * 128 * info["sm_clock_max_mhz"] * 1e6 / SASS_INSTR_PER_EVAL_K1
    g = torch.Generator(device=dev).manual_seed(0)
    res = {"gpu": info, "bound": "instruction issue, k = 1 kernels (SASS count, see tools/bench_knn.py)",
           "sass_instructions_per_eval_k1": SASS_INSTR_PER_EVAL_K1, "issue_bound_evals_per_s_k1": bound,
           "knn": [], "icp": {}}

    for N1, N2, k in ((100000, 100000, 1), (100000, 100000, 16), (2000, 100000, 8), (400000, 100000, 1),
                      (400000, 100000, 16)):
        ref = torch.rand(N1, 3, device=dev, generator=g)
        nbr = torch.rand(N2, 3, device=dev, generator=g)
        splits, _ = _knn._plan(1, N1, N2, k, ref)
        t = timed(lambda: pp.knn(ref, nbr, k=k), args.reps)
        base = timed(lambda: cdist_topk(ref, nbr, k), max(3, args.reps // 4))
        evals = N1 * N2
        row = {"N1": N1, "N2": N2, "D": 3, "k": k, "dtype": "float32", "splits": splits, "knn": t,
               "evals_per_s": evals / (t["median_ms"] * 1e-3),
               "share_of_issue_bound": evals / (t["median_ms"] * 1e-3) / bound if k == 1 else None,
               "cdist_topk_chunked": base, "speedup_vs_cdist_topk": base["median_ms"] / t["median_ms"]}
        res["knn"].append(row)
        print(json.dumps(row), flush=True)

    N = int(math.sqrt(REF_FORMULA_BYTES / 16))
    N = N - N % 1000
    ref = torch.rand(N, 3, device=dev, generator=g)
    nbr = torch.rand(N, 3, device=dev, generator=g)
    t_ref = timed(lambda: reference_formula(ref, nbr, 1), 3)
    torch.cuda.empty_cache()
    t_knn = timed(lambda: pp.knn(ref, nbr, k=1), args.reps)
    res["reference_formula"] = {"N1": N, "N2": N, "k": 1, "largest_size_within_budget": N,
                                "budget_bytes": REF_FORMULA_BYTES, "reference_formula": t_ref, "knn": t_knn,
                                "speedup": t_ref["median_ms"] / t_knn["median_ms"]}
    print(json.dumps(res["reference_formula"]), flush=True)
    del ref, nbr
    torch.cuda.empty_cache()

    B, n, iters = 8, 100000, 30
    src = torch.rand(B, n, 3, device=dev, generator=g) * torch.tensor([10.0, 10.0, 2.0], device=dev)
    tf = pp.randn_SE3(B, sigma=0.05, device=dev)
    tgt = tf.unsqueeze(-2).Act(src)
    splits, _ = _knn._plan(B, n, n, 1, src)
    icp = pp.module.ICP(stepper=pp.utils.ReduceToBason(steps=iters, patience=10 ** 9, tol=-1.0))
    t = timed(lambda: icp(src, tgt), max(3, args.reps // 4))
    evals = B * n * n * iters
    res["icp"] = {"B": B, "N": n, "iterations": iters, "dtype": "float32", "splits": splits, "icp": t,
                  "per_iteration_ms": t["median_ms"] / iters, "evals_per_s": evals / (t["median_ms"] * 1e-3),
                  "share_of_issue_bound": evals / (t["median_ms"] * 1e-3) / bound}
    print(json.dumps(res["icp"]), flush=True)
    res["measured_at"] = time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
