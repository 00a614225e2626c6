"""Throughput of the decoders and of the Sinkhorn EMD next to the point / latent loops (tracked numbers the round-1 review asked
for): FoldingDecoder (PointNetVAE.decode, networks.py:1449-1509) on the tcgen05 split-precision path, and
earth_mover_distance_gpu (metrics.py:94-158) on 2048-point clouds (one subprocess each)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def folding():
    import torch
    import pcd_b200
    from oracle import pointdiff_oracle as O
    NP = 2048
    fsd = O.make_synthetic_folding_checkpoint(num_points=NP)
    vae = pcd_b200.PointNetVAE(NP)
    vae.load_state_dict({k[len("vae."):]: v for k, v in fsd.items()}, strict=False)
    vae = vae.eval().cuda()
    g = torch.Generator().manual_seed(3)
    zc = torch.randn(2, 256, generator=g)
    err = float((vae.decode(zc.cuda()).cpu() - O.folding_decode(fsd, zc)).norm() / O.folding_decode(fsd, zc).norm())
    for B in (128, 1024):
        z = torch.randn(B, 256, generator=g).cuda()
        ms, out = timed(lambda: vae.decode(z), 5)
        flops = 2.0 * B * 1024 * (2 * (512 * 512 + 3 * 512 + 512 * 3) + 9 * 2) + 2.0 * 3 * B * 1024 * NP
        print(json.dumps({"what": "FoldingDecoder.decode -> 2048 pts", "path": "tcgen05 fp16 hi+lo, 3 passes",
                          "batch": B, "ms": ms, "latents_per_s": B / ms * 1e3, "algorithmic_tflops": flops / ms / 1e9,
                          "rel_l2_vs_oracle_b2": err, "finite": bool(torch.isfinite(out).all())}), flush=True)


def emd():
    import torch
    import pcd_b200
    g = torch.Generator().manual_seed(4)
    for B in (16, 128):
        x = (torch.randn(B, 2048, 3, generator=g) * torch.rand(B, 1, 3, generator=g)).cuda()
        y = (torch.randn(B, 2048, 3, generator=g) * torch.rand(B, 1, 3, generator=g)).cuda()
        ms, (val, iters) = timed(lambda: pcd_b200._lib.sinkhorn_emd(x, y, 1e-2, 1e-5, 100), 2)
        ev = 2.0 * B * 2048 * 2048 * iters
        print(json.dumps({"what": "earth_mover_distance_gpu (Sinkhorn), 2048 x 2048 points per pair", "pairs": B, "iterations": iters, "ms": ms,
                          "pairs_per_s": B / ms * 1e3, "cost_evals_per_s": ev / ms * 1e3, "mean_emd": float(val.mean())}), flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1:
        {"folding": folding, "emd": emd}[sys.argv[1]]()
    else:
        subprocess.run([sys.executable, __file__, "folding"], timeout=600)
        subprocess.run([sys.executable, __file__, "emd"], timeout=600)
