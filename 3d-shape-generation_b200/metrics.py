"""Chamfer core of the reference's metrics.py (:7-47), its Sinkhorn and exact EMD (:49-158) on the B200 kernels, plus the
set-level metrics (MMD / COV / 1-NNA over CD or EMD) built on the reference's per-pair semantics.

`chamfer_distance(x, y, scaling_factor=1e3)` keeps the reference signature and return type
(0-dim tensor; batched input -> one scalar averaged over the batch).
"""
from __future__ import annotations

import torch

from . import _lib


def chamfer_distance(x: torch.Tensor, y: torch.Tensor, scaling_factor: float = 1e3, *, return_indices: bool = False):
    """Reference metrics.py:23-47 (with normalize_to_cube :7-21 fused in)."""
    x = x.unsqueeze(0) if x.dim() == 2 else x
    y = y.unsqueeze(0) if y.dim() == 2 else y
    if return_indices:
        cd, ixy, iyx = _lib.chamfer_pairs(x, y, scaling_factor, return_indices=True)
        return cd.mean(), ixy, iyx
    return _lib.chamfer_pairs(x, y, scaling_factor).mean()


def chamfer_distance_per_pair(x: torch.Tensor, y: torch.Tensor, scaling_factor: float = 1e3) -> torch.Tensor:
    """cd[b] for each pair (x[b], y[b]) -- what the reference's per-sample loop computes
    (test_point_ddpm.py:85-86 -> metrics.py:172)."""
    return _lib.chamfer_pairs(x, y, scaling_factor)


def earth_mover_distance_gpu(x: torch.Tensor, y: torch.Tensor, epsilon: float = 1e-2, thresh: float = 1e-5, max_iter: int = 100,
                            scaling_factor: float = 1):
    """Reference metrics.py:94-158 (log-domain Sinkhorn "EMD"): same signature, 0-dim tensor averaged over
    the batch.  The [n, m] cost matrix is recomputed on the fly instead of materialised."""
    x = x.unsqueeze(0) if x.dim() == 2 else x
    y = y.unsqueeze(0) if y.dim() == 2 else y
    emd, _ = _lib.sinkhorn_emd(x, y, epsilon, thresh, max_iter, 1.0)
    return emd.mean() * scaling_factor


def earth_mover_distance_exact(x: torch.Tensor, y: torch.Tensor, *, return_assignment: bool = False):
    """Reference metrics.py:49-92 (`earth_mover_distance_cpu`) on the GPU: an optimal one-to-one matching of the two
    cube-normalised clouds under Euclidean distance, matched sum divided by 3 (the reference's divisor).  N != M matches
    min(N, M) pairs.  [N, 3] inputs are promoted to a batch of one; batched input -> the mean over pairs as a 0-dim float32
    device tensor.  Optimal for distances quantised to 2^-22 (within max(N, M) / 2^22 of the fp64 optimum per pair), at most
    4096 points per cloud.  return_assignment=True also returns the matched y index of every x, int32 [B, N] (-1: unmatched)."""
    x = x.unsqueeze(0) if x.dim() == 2 else x
    y = y.unsqueeze(0) if y.dim() == 2 else y
    if return_assignment:
        emd, assign = _lib.emd_exact(x, y, return_assignment=True)
        return emd.mean(), assign
    return _lib.emd_exact(x, y).mean()


_WARNED = set()


def _warn_once(key: str, msg: str) -> None:
    if key not in _WARNED:
        _WARNED.add(key)
        import warnings
        warnings.warn(msg, stacklevel=3)


def voxelize(points: torch.Tensor, voxel_resolution: int = 32) -> torch.Tensor:
    """Reference utils.py:488-509 (occupancy scatter, truncating `.long()` cast, clamp to the grid) as device torch ops:
    [B, N, 3] -> [B, R, R, R] in {0, 1}.  Plumbing for `compute_metrics`' third value, not a hot path."""
    points = points.unsqueeze(0) if points.dim() == 2 else points
    idx = ((points + 1) * (voxel_resolution - 1) / 2).long().clamp(0, voxel_resolution - 1)
    B, R = points.size(0), voxel_resolution
    flat = (idx[..., 0] * R + idx[..., 1]) * R + idx[..., 2]
    vox = torch.zeros(B, R * R * R, device=points.device)
    vox.scatter_(1, flat, 1.0)
    return vox.view(B, R, R, R)


def compute_metrics(generated_samples, reference_samples, use_approximate_gpu_emd=False, *, emd_fn=None, recon_fn=None):
    """Reference metrics.py:160-183 boundary: returns three 0-dim tensors (avg_cd, avg_emd, recon_loss), so the reference's
    callers (`avg_emd += emd`, `f"{emd:.3f}"`, test_point_ddpm.py:85-114) run unchanged.

    * Chamfer: the B200 kernels.
    * EMD: `use_approximate_gpu_emd=True` -> the Sinkhorn EMD on the B200 kernels (metrics.py:94-158).  The reference's default is
      the exact assignment (SciPy Hungarian, metrics.py:49-92).  Without an `emd_fn` the default evaluates the Sinkhorn EMD and
      says so once -- its values are NOT comparable with the exact EMD (5.995 vs 44.307 on the reference's own unit-test inputs).
      Pass `emd_fn=pcd_b200.earth_mover_distance_exact` for the exact value on the GPU.
    * recon_loss: binary cross-entropy between the two 32^3 occupancy grids (metrics.py:181), same expression as the reference.
    """
    avg_cd = chamfer_distance(generated_samples, reference_samples)
    if emd_fn is not None:
        avg_emd = emd_fn(generated_samples, reference_samples)
    else:
        if not use_approximate_gpu_emd:
            _warn_once("emd", "pcd_b200.compute_metrics: returning the Sinkhorn EMD (earth_mover_distance_gpu), not the reference's "
                              "default exact EMD -- pass emd_fn=pcd_b200.earth_mover_distance_exact for the exact value")
        avg_emd = earth_mover_distance_gpu(generated_samples, reference_samples)
    if recon_fn is not None:
        recon = recon_fn(generated_samples, reference_samples)
    else:
        recon = torch.nn.functional.binary_cross_entropy(voxelize(generated_samples), voxelize(reference_samples))
    return avg_cd, avg_emd, recon


def chamfer_matrix(G: torch.Tensor, R: torch.Tensor, scaling_factor: float = 1e3) -> torch.Tensor:
    """D[i, j] = chamfer_distance(G[i], R[j])."""
    return _lib.chamfer_matrix(G, R, scaling_factor)


_EMD_MATRIX_CHUNK = 4096   # pairs per kernel call: bounds the gathered copies of the clouds (2 x 100 MB at 2048 points)


def emd_matrix(G: torch.Tensor, R: torch.Tensor, scaling_factor: float = 1.0) -> torch.Tensor:
    """D[i, j] = earth_mover_distance_exact(G[i], R[j]) * scaling_factor; every cloud has the same point count.  A set against
    itself (same tensor) evaluates i <= j only and mirrors it, so emd_matrix(X, X) is symmetric bit for bit."""
    assert G.shape[1] == R.shape[1], "all clouds must have the same number of points"
    nG, nR = G.shape[0], R.shape[0]
    self_mode = G.data_ptr() == R.data_ptr() and G.shape == R.shape and G.stride() == R.stride()
    if self_mode:
        ii, jj = torch.triu_indices(nG, nG, device=G.device)
    else:
        ii = torch.arange(nG, device=G.device).repeat_interleave(nR)
        jj = torch.arange(nR, device=G.device).repeat(nG)
    step = _EMD_MATRIX_CHUNK
    vals = torch.cat([_lib.emd_exact(G[ii[k:k + step]], R[jj[k:k + step]], scaling_factor)
                      for k in range(0, ii.numel(), step)]) if ii.numel() else torch.empty(0, device=G.device)
    out = torch.empty(nG, nR, device=G.device, dtype=torch.float32)
    out[ii, jj] = vals
    if self_mode:
        out[jj, ii] = vals
    return out


def set_metrics_from_matrices(D_gr: torch.Tensor, D_gg: torch.Tensor, D_rr: torch.Tensor) -> dict:
    """MMD-CD, COV-CD, 1-NNA-CD (Achlioptas et al. 2018; Yang et al. 2019).  Not in the reference
    (SURVEY 0.8); tiny reductions over the CD matrices, done with torch ops on the device."""
    nG, nR = D_gr.shape
    mmd = D_gr.min(dim=0)[0].mean()
    cov = torch.unique(D_gr.argmin(dim=1)).numel() / nR
    full = torch.cat([torch.cat([D_gg, D_gr], dim=1), torch.cat([D_gr.t(), D_rr], dim=1)], dim=0).clone()
    full.fill_diagonal_(float("inf"))
    nn_idx = full.argmin(dim=1)
    label = torch.cat([torch.zeros(nG, device=full.device), torch.ones(nR, device=full.device)])
    acc = (label[nn_idx] == label).float().mean()
    return {"mmd_cd": float(mmd), "cov_cd": float(cov), "1nna_cd": float(acc)}


_INF = float("inf")


def _keys(values: torch.Tensor, index: torch.Tensor) -> torch.Tensor:
    """(non-negative fp32 value, index) -> one int64 whose order is (value, index): min over keys = first argmin."""
    bits = values.contiguous().view(torch.int32).to(torch.int64)          # >= 0 floats: the bit pattern is order preserving
    return (bits << 32) | index.to(torch.int64)


def _gather_uneven(local: torch.Tensor):
    """all_gather of per-rank row blocks whose sizes may differ (shard_range leaves a remainder): counts first, pad to the
    largest block, gather, slice.  Returns (concatenated tensor, first global row of this rank)."""
    import torch.distributed as dist
    W, rank = dist.get_world_size(), dist.get_rank()
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
    counts = [torch.zeros_like(n) for _ in range(W)]
    dist.all_gather(counts, n)
    counts = [int(c) for c in counts]
    cap = max(counts)
    pad = torch.zeros((cap,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    parts = [torch.empty_like(pad) for _ in range(W)]
    dist.all_gather(parts, pad)
    return torch.cat([p[:c] for p, c in zip(parts, counts)]), sum(counts[:rank])


def evaluate_sets(G_local: torch.Tensor, R_local: torch.Tensor, scaling_factor: float = 1e3, *, metric: str = "cd", matrix_fn=None,
                  tile: int = None) -> dict:
    """MMD-CD / COV-CD / 1-NNA-CD (Achlioptas et al. 2018; Yang et al. 2019 -- not in the reference, SURVEY 0.8) for generated /
    reference clouds sharded over ranks (one process per GPU; shards may be uneven).

    metric="emd" sweeps with `emd_matrix` instead and returns mmd_emd / cov_emd / 1nna_emd with the same definitions, in the
    reference's EMD unit (`scaling_factor` applies to CD only).  `matrix_fn(A, B, scale)` overrides the matrix function.

    One exchange step: NCCL all-gather of both sets.  The three CD matrices are never assembled: they are cut into `tile` x `tile`
    blocks, dealt round-robin to the ranks, and each block is reduced on the spot to row / column minima.  D_gg and D_rr are
    symmetric (bit for bit: the fused kernel evaluates each point pair once), so only their upper-triangle blocks are computed --
    the sweep costs 2x the G x R pair count (+ n) instead of 3x.  What crosses ranks afterwards is five [n] vectors
    (all_reduce(MIN)), as SURVEY 8(e) sketches.  Ties follow `argmin` on the assembled matrices (first index wins)."""
    import torch.distributed as dist
    if metric not in ("cd", "emd"):
        raise ValueError("metric must be 'cd' or 'emd'")
    if metric == "emd":
        cm, scaling_factor = emd_matrix, 1.0
    else:
        cm = chamfer_matrix
    cm = cm if matrix_fn is None else matrix_fn   # injectable so the gloo/CPU test can exercise the exchange
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    if multi:
        W, rank = dist.get_world_size(), dist.get_rank()
        G, _ = _gather_uneven(G_local.contiguous())
        R, _ = _gather_uneven(R_local.contiguous())
    else:
        W, rank, G, R = 1, 0, G_local, R_local
    nG, nR, dev = G.shape[0], R.shape[0], G.device
    if tile is None:      # ~32 blocks per side, 128..512 clouds per block (a diagonal block costs half: chamfer_matrix(X, X) mirrors its upper triangle)
        tile = min(512, max(128, -(-max(nG, nR) // 32 // 64) * 64))
    big = torch.iinfo(torch.int64).max
    gr_row = torch.full((nG,), big, dtype=torch.int64, device=dev)      # per g: min_r (D_gr, r) -> COV and 1-NNA
    gr_col = torch.full((nR,), _INF, device=dev)                        # per r: min_g D_gr      -> MMD and 1-NNA
    gg = torch.full((nG,), _INF, device=dev)                            # per g: min_{g' != g} D_gg
    rr = torch.full((nR,), _INF, device=dev)
    job = 0
    for i0 in range(0, nG, tile):
        for j0 in range(0, nR, tile):
            job += 1
            if (job - 1) % W != rank:
                continue
            D = cm(G[i0:i0 + tile], R[j0:j0 + tile], scaling_factor)
            v, a = D.min(dim=1)
            gr_row[i0:i0 + tile] = torch.minimum(gr_row[i0:i0 + tile], _keys(v, a + j0))
            gr_col[j0:j0 + tile] = torch.minimum(gr_col[j0:j0 + tile], D.min(dim=0)[0])
    for X, acc in ((G, gg), (R, rr)):
        n = X.shape[0]
        for i0 in range(0, n, tile):
            for j0 in range(i0, n, tile):                                # upper triangle of blocks only
                job += 1
                if (job - 1) % W != rank:
                    continue
                D = cm(X[i0:i0 + tile], X[j0:j0 + tile], scaling_factor)
                if i0 == j0:
                    D = D.clone()
                    D.fill_diagonal_(_INF)
                acc[i0:i0 + tile] = torch.minimum(acc[i0:i0 + tile], D.min(dim=1)[0])
                if i0 != j0:                                             # the mirrored block, by symmetry
                    acc[j0:j0 + tile] = torch.minimum(acc[j0:j0 + tile], D.min(dim=0)[0])
    if multi:
        for v in (gr_row, gr_col, gg, rr):
            dist.all_reduce(v, op=dist.ReduceOp.MIN)
    gr_row_val = (gr_row >> 32).to(torch.int32).view(torch.float32)
    nn_ref = gr_row & 0xFFFFFFFF
    mmd = gr_col.mean()
    cov = torch.unique(nn_ref).numel() / nR
    # 1-NNA on the concatenation [G | R]: a g row's nearest neighbour is another g unless some r is strictly closer (G columns
    # come first in the assembled matrix, so argmin breaks ties towards G for every row)
    correct = (gg <= gr_row_val).sum() + (rr < gr_col).sum()
    return {"mmd_" + metric: float(mmd), "cov_" + metric: float(cov), "1nna_" + metric: int(correct) / float(nG + nR)}
