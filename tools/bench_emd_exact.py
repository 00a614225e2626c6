"""Exact EMD throughput: the auction kernel (pcd_emd_exact) on one GPU against SciPy's linear_sum_assignment on the host, in one run.

    python tools/bench_emd_exact.py [--out profiles/emd_exact_bench.jsonl]

Prints one JSON line per measurement (and appends them to --out when given): GPU pairs/s at 2048 x 2048 points for batches of
16, 148 and 592 pairs (CUDA events after one warm-up call), the host rate of the SciPy restatement (tests/exact_emd_scipy.py)
in this single process on a few pairs, and the card name, power limit and host core count.  Inputs are seeded anisotropic Gaussian clouds.  Batch 16 is
the per-pair loop of the reference's evaluation script; it occupies 16 of the card's SMs (one CTA per pair)."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import exact_emd_scipy as S  # noqa: E402
import pcd_b200  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "host_cores": os.cpu_count()}


def clouds(seed: int, B: int, N: int, shift: float = 0.0) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, N, 3, generator=g) * (0.2 + torch.rand(B, 1, 3, generator=g)) + shift


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2048)
    ap.add_argument("--batches", type=int, nargs="+", default=[16, 148, 592])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-pairs", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the GPU rate needs a CUDA device"
    info = card()
    lines = []
    N = a.n
    for B in a.batches:
        x, y = clouds(B, B, N).cuda(), clouds(B + 1, B, N, 0.1).cuda()
        emd = pcd_b200._lib.emd_exact(x, y)                 # warm-up (module load, smem attribute)
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(a.reps):
            emd = pcd_b200._lib.emd_exact(x, y)
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / a.reps
        lines.append({"what": "pcd_emd_exact (auction, one CTA per pair)", "n": N, "pairs": B, "ms_per_call": round(ms, 3),
                      "pairs_per_s": round(B / ms * 1e3, 2), "reps": a.reps, "mean_emd": float(emd.mean()), **info})
        print(json.dumps(lines[-1]), flush=True)
    # host: the SciPy restatement (cdist fp64 + linear_sum_assignment) in this single process
    x, y = clouds(16, a.host_pairs, N), clouds(17, a.host_pairs, N, 0.1)
    t = time.perf_counter()
    want = S.exact_emd(x, y, per_pair=True)
    s = time.perf_counter() - t
    got = pcd_b200._lib.emd_exact(x.cuda(), y.cuda()).cpu().double()
    lines.append({"what": "SciPy linear_sum_assignment (tests/exact_emd_scipy.py), single process", "n": N, "pairs": a.host_pairs,
                  "s": round(s, 3), "pairs_per_s": round(a.host_pairs / s, 3),
                  "max_rel_diff_gpu_vs_scipy": float(((got - want).abs() / want).max()), **info})
    print(json.dumps(lines[-1]), flush=True)
    b16 = [l for l in lines if l.get("pairs") == 16 and "auction" in l["what"]]
    if b16:
        print(json.dumps({"what": "batch-16 GPU rate / host SciPy rate", "ratio": round(b16[0]["pairs_per_s"] / lines[-1]["pairs_per_s"], 1)}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
