"""GPU: non-finite and degenerate clouds through every metric kernel that shares `cloud_norm_kernel`, against the reference's
semantics as the oracle reproduces them on CPU.

`normalize_to_cube` (metrics.py:7-21) turns a cloud with a NaN or +-inf coordinate, a centre that overflows, or all points equal
(one point included) into NaN: torch.max / min / abs().max() propagate NaN, and inf - inf enters the scale.  What follows:
* Chamfer (pair kernels, values and index paths, fused and directional; all-pairs and self matrices) and exact EMD evaluate each
  pair on its own: the bad pair is NaN, and every other pair equals, bit for bit, the same pair evaluated in a batch without the
  bad cloud.
* Sinkhorn takes ONE cost maximum and ONE convergence test over the batch (metrics.py:124, :148-151): every pair is NaN and the
  loop runs exactly max_iter iterations."""
import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O

pytestmark = pytest.mark.gpu
NAN, INF = float("nan"), float("inf")


def _make_bad(case: str, x: torch.Tensor) -> torch.Tensor:
    """A copy of x [3, N, 3] whose cloud 1 is bad (the one-point case keeps the first point of every cloud: all pairs are bad)."""
    x = x.clone()
    if case.startswith("nan_"):
        x[1, 137, "xyz".index(case[-1])] = NAN
    elif case == "inf_y":
        x[1, 137, 1] = INF
    elif case == "neg_inf_z":
        x[1, 137, 2] = -INF
    elif case == "pos_and_neg_inf_y":
        x[1, 17, 1], x[1, 137, 1] = INF, -INF
    elif case == "all_points_equal":
        x[1] = 0.25
    elif case == "one_point":
        x = x[:, :1].contiguous()
    elif case == "centre_overflows_y":            # finite, but max + min = inf
        x[1, :, 1] = 3e38 * (0.9 + 0.1 * torch.rand(x.shape[1], generator=torch.Generator().manual_seed(5)))
    else:
        raise ValueError(case)
    return x


CASES = ["nan_x", "nan_y", "nan_z", "inf_y", "neg_inf_z", "pos_and_neg_inf_y", "all_points_equal", "one_point",
         "centre_overflows_y"]


def _clouds(seed, B, N, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, N, 3, generator=g) * (0.2 + torch.rand(B, 1, 3, generator=g)) + shift


def _bad_pairs(x, y):
    """Pairs whose reference normalisation is not finite."""
    fin = lambda c: torch.isfinite(O.normalize_to_cube(c)).flatten(1).all(1)
    return ~(fin(x) & fin(y))


def _check_chamfer_pairs(x, y, bad):
    good = (~bad).nonzero().squeeze(1)
    cd = pcd_b200._lib.chamfer_pairs(x.cuda(), y.cuda(), 1e3).cpu()
    cdi, ixy, iyx = (t.cpu() for t in pcd_b200._lib.chamfer_pairs(x.cuda(), y.cuda(), 1e3, return_indices=True))
    assert torch.equal(torch.isnan(cd), bad) and torch.equal(torch.isnan(cdi), bad), (cd, cdi, bad)
    if good.numel():
        assert torch.equal(cd[good], pcd_b200._lib.chamfer_pairs(x[good].cuda(), y[good].cuda(), 1e3).cpu())
        ref = [t.cpu() for t in pcd_b200._lib.chamfer_pairs(x[good].cuda(), y[good].cuda(), 1e3, return_indices=True)]
        assert torch.equal(cdi[good], ref[0]) and torch.equal(ixy[good], ref[1]) and torch.equal(iyx[good], ref[2])


def _check_chamfer_matrix(G, R, bad_g):
    """G has the bad cloud, R [2, N, 3] is finite: all pairs, then G against itself (the triangle path)."""
    good = (~bad_g).nonzero().squeeze(1)
    D = pcd_b200.chamfer_matrix(G.cuda(), R.cuda()).cpu()
    assert torch.equal(torch.isnan(D), bad_g[:, None].expand_as(D)), D
    S = pcd_b200.chamfer_matrix(G.cuda(), G.cuda()).cpu()
    assert torch.equal(torch.isnan(S), bad_g[:, None] | bad_g[None, :]), S
    if good.numel():
        Gg = G[good].cuda()
        assert torch.equal(D[good], pcd_b200.chamfer_matrix(Gg, R.cuda()).cpu())
        assert torch.equal(S[good][:, good], pcd_b200.chamfer_matrix(Gg, Gg).cpu())


@pytest.mark.parametrize("case", CASES)
def test_nonfinite_cloud_small_shape(case):
    """300 x 200 points: the fused pair kernel, the index passes, the fused matrix kernels, Sinkhorn and exact EMD."""
    x, y = _make_bad(case, _clouds(1, 3, 300)), _clouds(2, 3, 200, 0.1)
    bad = _bad_pairs(x, y)
    assert bool(bad[1]) and (case == "one_point" or not bool(bad[[0, 2]].any()))
    # the reference's semantics, on CPU
    assert torch.equal(torch.isnan(O.chamfer_pairs(x, y)[0]), bad)
    want, it_want = O.sinkhorn_emd(x, y, epsilon=0.1, thresh=1e-5, max_iter=30, exact=True, per_pair=True)
    assert bool(torch.isnan(want).all()) and it_want == 30
    for a, b in ((x, y), (y, x)):                 # the bad cloud as queries, then as targets
        _check_chamfer_pairs(a, b, bad)
        # Sinkhorn: one bad pair poisons the batch maximum and the convergence test (the finite pairs alone stop after ~5)
        got, it = pcd_b200._lib.sinkhorn_emd(a.cuda(), b.cuda(), 0.1, 1e-5, 30)
        assert bool(torch.isnan(got).all()) and it == 30, (got, it)
        # exact EMD
        emd, assign = pcd_b200._lib.emd_exact(a.cuda(), b.cuda(), return_assignment=True)
        emd, assign = emd.cpu(), assign.cpu()
        assert torch.equal(torch.isnan(emd), bad) and bool((assign[bad] == -1).all()), emd
        good = (~bad).nonzero().squeeze(1)
        if good.numel():
            ref, ref_assign = pcd_b200._lib.emd_exact(a[good].cuda(), b[good].cuda(), return_assignment=True)
            assert torch.equal(emd[good], ref.cpu()) and torch.equal(assign[good], ref_assign.cpu())
    _check_chamfer_matrix(x, _clouds(3, 2, x.shape[1], 0.2), bad)


@pytest.mark.parametrize("case", [c for c in CASES if c != "one_point"])
def test_nonfinite_cloud_directional_shape(case):
    """6500 x 6400 points: beyond the fused kernel's 200 KB of shared memory (4500 x 4100 still fits, in 137 KB), values take the
    directional passes and 6500-point matrices the two-pass matrix kernel."""
    x, y = _make_bad(case, _clouds(11, 3, 6500)), _clouds(12, 3, 6400, 0.1)
    bad = _bad_pairs(x, y)
    assert bad.tolist() == [False, True, False]
    for a, b in ((x, y), (y, x)):
        _check_chamfer_pairs(a, b, bad)
    _check_chamfer_matrix(x, _clouds(13, 2, 6500, 0.2), bad)
