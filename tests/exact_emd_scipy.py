"""CPU reference for the exact EMD (the original project's `earth_mover_distance_cpu`, metrics.py:49-92), restated with SciPy.
Imported by the exact-EMD tests and by tools/bench_emd_exact.py; not a test module itself."""
import numpy as np
import torch
from scipy.optimize import linear_sum_assignment
from scipy.spatial.distance import cdist

from oracle.pointdiff_oracle import normalize_to_cube


def exact_emd(x: torch.Tensor, y: torch.Tensor, per_pair: bool = False, return_assignment: bool = False):
    """Per pair: cube-normalise (fp32), Euclidean distances in fp64 (SciPy cdist), optimal assignment (SciPy
    linear_sum_assignment; N != M matches min(N, M) pairs), matched sum / 3 (the original divides by x_pc.shape[1]).
    Batched input -> the mean over pairs as float32 (per_pair=True: the float64 values [B]).
    return_assignment=True also returns the matched y index of every x, int64 [B, N] (-1: unmatched)."""
    x = x.unsqueeze(0) if x.dim() == 2 else x
    y = y.unsqueeze(0) if y.dim() == 2 else y
    xn, yn = normalize_to_cube(x.float()).double().numpy(), normalize_to_cube(y.float()).double().numpy()
    vals = torch.empty(x.shape[0], dtype=torch.float64)
    assign = torch.full((x.shape[0], x.shape[1]), -1, dtype=torch.int64)
    for b in range(x.shape[0]):
        C = cdist(xn[b], yn[b])
        r, c = linear_sum_assignment(C)
        vals[b] = float(C[r, c].sum()) / 3
        assign[b, torch.from_numpy(r)] = torch.from_numpy(c.astype(np.int64))
    out = vals if per_pair else vals.mean().float()
    return (out, assign) if return_assignment else out
