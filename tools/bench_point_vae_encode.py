"""Point-VAE encoder (SimplePointNetVAE.encode): per-layer parity against the oracle, encode time, clouds/s and useful TFLOP/s,
per-layer ms and TFLOP/s, and eager PyTorch on the same GPU for context.
    python tools/bench_point_vae_encode.py [--batches 16,128,512] [--points 2048] [--precisions bf16x3,f16mix,bf16,f16]
Prints one JSON line per precision.  Input clouds are Gaussian (the time does not depend on the values)."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pcd_b200  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tests"))
import point_vae_encoder_oracle as P  # noqa: E402  (checker and eager baseline)


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def useful_gflop_per_cloud(n_points):
    """Shape-derived FLOPs of one encode: the 12 per-point convs (1,737,088 per point) and the heads (524,288 per cloud)."""
    per_point = 0
    for ci, co in ((3, 64), (64, 128), (128, 256), (256, 512)):
        per_point += 2 * (ci * co + 2 * co * co)
    return (per_point * n_points + 2 * (512 * 256 + 2 * 256 * 256)) * 1e-9


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for i in range(reps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(reps))[reps // 2]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="16,128,512")
    ap.add_argument("--points", type=int, default=2048)
    ap.add_argument("--parity-batch", type=int, default=3)
    ap.add_argument("--precisions", default="bf16x3,f16mix,bf16,f16")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--eager", type=int, default=1, help="also time the eager PyTorch encoder")
    args = ap.parse_args()
    batches = [int(b) for b in args.batches.split(",")]
    N = args.points
    sd = P.make_synthetic_point_vae_encoder_checkpoint()
    g = torch.Generator().manual_seed(3)
    xp = torch.randn(args.parity_batch, N, 3, generator=g)
    taps = {}
    t0 = time.time()
    want_mu, want_lv = P.point_vae_encode(sd, xp, taps=taps)
    cpu_s = time.time() - t0
    gfl = useful_gflop_per_cloud(N)
    xs = {B: torch.randn(B, N, 3, generator=g).cuda() for B in batches}
    eager = {}
    if args.eager:
        sdc = {k: v.cuda() for k, v in sd.items()}
        for name, tf32 in (("eager_fp32_strict", False), ("eager_torch_default", None)):
            old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
            if tf32 is not None:
                torch.backends.cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = tf32
            with torch.no_grad():
                eager[name] = {str(B): round(timed(lambda: P.point_vae_encode(sdc, xs[B]), 3, 1), 3) for B in batches}
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        del sdc
        torch.cuda.empty_cache()
    info = gpu_info()
    for prec in args.precisions.split(","):
        eng = pcd_b200.PointEncoderEngine(sd, torch.device("cuda", 0), prec)
        errs = {str(i): rel_l2(eng.tap(xp.cuda(), i), taps[i]) for i in range(14)}
        mu, lv = eng.encode(xp.cuda())
        res = {"precision": prec, "gpu": info, "points": N, "useful_gflop_per_cloud": round(gfl, 4),
               "parity": {"batch": args.parity_batch, "tap_rel_l2": errs, "mu_rel_l2": rel_l2(mu, want_mu), "logvar_rel_l2": rel_l2(lv, want_lv)},
               "cpu_oracle_s_per_cloud": cpu_s / args.parity_batch, "encode": {}}
        for B in batches:
            ms = timed(lambda: eng.encode(xs[B]), args.reps)
            res["encode"][str(B)] = {"ms": round(ms, 3), "clouds_per_s": round(B / ms * 1e3, 1), "useful_tflops": round(gfl * B / ms, 1)}
            if args.eager:
                res["encode"][str(B)].update({k: v[str(B)] for k, v in eager.items()})
        prof = eng.profile(xs[batches[-1]])
        res["layers_batch"] = batches[-1]
        res["layers"] = {n: {"ms": round(m, 4), "tflops": round(fl / m * 1e-9, 1) if m > 0 else 0} for n, m, fl in prof}
        print(json.dumps(res), flush=True)
        eng.close()
        del eng
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
