"""GPU: Chamfer kernels through the C ABI against the reference golden values and the oracle.

Tolerances: the reference's torch.cdist takes the matmul path (|x|^2+|y|^2-2xy), whose own error
vs fp64 is 8.6e-6 absolute on unit-cube clouds (SURVEY H9); our kernel uses direct differences
(more accurate).  Values: rtol 2e-5 against the reference; 2e-6 against the exact oracle.
Nearest-neighbour indices: bit-exact against the exact (direct-difference) oracle except where
the two best candidates are within 4 ulp of each other."""
import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O
from conftest import same_set_metrics

pytestmark = pytest.mark.gpu


def test_reference_unit_test_inputs(golden):
    """units.py:7-26: seed-0 randn(1,994,3) vs randn(1,948,3); the reference asserts 0 <= CD <= 200."""
    cd = pcd_b200.chamfer_distance(golden["cd.units.x"].cuda(), golden["cd.units.y"].cuda())
    assert cd.dim() == 0 and cd.is_cuda
    assert 0.0 <= float(cd) <= 200.0
    assert abs(float(cd) - 142.71389770507812) < 142.7 * 2e-5
    # 2-D inputs are promoted to a batch of one (metrics.py:35-36)
    cd2 = pcd_b200.chamfer_distance(golden["cd.units.x"][0].cuda(), golden["cd.units.y"][0].cuda())
    assert float(cd2) == float(cd)


def test_batched_ragged_vs_reference_golden(golden):
    x, y = golden["cd.batch.x"].cuda(), golden["cd.batch.y"].cuda()     # N=512 vs M=300
    assert abs(float(pcd_b200.chamfer_distance(x, y)) - float(golden["cd.batch.value"])) < 2e-5 * float(golden["cd.batch.value"])
    pp = pcd_b200.chamfer_distance_per_pair(x, y).cpu()
    assert torch.allclose(pp, golden["cd.batch.per_pair"], rtol=2e-5)


def test_values_and_indices_vs_exact_oracle():
    g = torch.Generator().manual_seed(41)
    x = torch.randn(8, 2048, 3, generator=g) * torch.rand(8, 1, 3, generator=g)
    y = torch.randn(8, 2048, 3, generator=g) * torch.rand(8, 1, 3, generator=g) + 0.1
    cd_ref, ixy_ref, iyx_ref = O.chamfer_pairs(x, y)
    cd, ixy, iyx = pcd_b200._lib.chamfer_pairs(x.cuda(), y.cuda(), 1e3, return_indices=True)
    assert torch.allclose(cd.cpu(), cd_ref, rtol=2e-6)
    xn, yn = O.normalize_to_cube(x), O.normalize_to_cube(y)
    for got, want, q, t in ((ixy.cpu().long(), ixy_ref, xn, yn), (iyx.cpu().long(), iyx_ref, yn, xn)):
        diff = got != want
        if diff.any():
            # any disagreement must be a near-tie between the two candidates
            b, i = diff.nonzero(as_tuple=True)
            d_got = (q[b, i] - t[b, got[b, i]]).norm(dim=-1)
            d_want = (q[b, i] - t[b, want[b, i]]).norm(dim=-1)
            assert torch.allclose(d_got, d_want, rtol=5e-7, atol=0), "index flip that is not a tie"
        assert float(diff.float().mean()) < 1e-3


def test_properties_symmetry_identity_scaling():
    g = torch.Generator().manual_seed(42)
    x, y = torch.randn(3, 700, 3, generator=g).cuda(), torch.randn(3, 333, 3, generator=g).cuda()
    a, b = pcd_b200.chamfer_distance_per_pair(x, y), pcd_b200.chamfer_distance_per_pair(y, x)
    assert torch.allclose(a, b, rtol=1e-6)
    assert float(pcd_b200.chamfer_distance_per_pair(x, x).abs().max()) == 0.0       # exact path: CD(x,x) = 0
    # cube normalisation makes CD invariant to translation and uniform scale
    c = pcd_b200.chamfer_distance_per_pair(x * 3.0 + 5.0, y * 0.5 - 2.0)
    assert torch.allclose(a, c, rtol=1e-4)
    assert torch.allclose(pcd_b200.chamfer_distance_per_pair(x, y, 1.0) * 1e3, a, rtol=1e-6)


def test_degenerate_cloud_gives_nan_like_reference():
    x = torch.ones(1, 16, 3).cuda()          # all points equal -> scale 0 -> 0/0 (metrics.py:19-20)
    y = torch.randn(1, 16, 3).cuda()
    assert torch.isnan(pcd_b200.chamfer_distance(x, y))
    assert torch.isnan(O.chamfer_distance(x.cpu(), y.cpu()))


def test_nan_coordinate_poisons_the_cloud_like_reference():
    """torch.max / torch.min propagate NaN (metrics.py:17-18): one NaN coordinate anywhere in a cloud makes its distance NaN, in
    the pair kernels (values and indices paths) and in the matrix kernel; the other clouds of the batch are unaffected."""
    g = torch.Generator().manual_seed(44)
    x, y = torch.randn(3, 300, 3, generator=g), torch.randn(3, 200, 3, generator=g)
    x[1, 137, 2] = float("nan")            # not element 0
    want = O.chamfer_pairs(x, y)[0]
    assert bool(torch.isnan(want[1])) and not bool(torch.isnan(want[0])) and not bool(torch.isnan(want[2]))
    got = pcd_b200.chamfer_distance_per_pair(x.cuda(), y.cuda()).cpu()
    assert torch.equal(torch.isnan(got), torch.isnan(want)) and torch.allclose(got[[0, 2]], want[[0, 2]], rtol=3e-6)
    got_i = pcd_b200._lib.chamfer_pairs(x.cuda(), y.cuda(), 1e3, return_indices=True)[0].cpu()
    assert torch.equal(torch.isnan(got_i), torch.isnan(want))
    D = pcd_b200.chamfer_matrix(x.cuda(), torch.randn(3, 300, 3, generator=g).cuda()).cpu()      # the matrix kernel: equal point counts
    assert bool(torch.isnan(D[1]).all()) and not bool(torch.isnan(D[[0, 2]]).any())
    assert torch.isnan(pcd_b200.chamfer_distance(x.cuda(), y.cuda())) and torch.isnan(O.chamfer_distance(x, y))


def test_matrix_vs_oracle_and_set_metrics():
    g = torch.Generator().manual_seed(43)
    G = torch.randn(6, 512, 3, generator=g) * torch.rand(6, 1, 3, generator=g)
    R = torch.randn(5, 512, 3, generator=g) * torch.rand(5, 1, 3, generator=g)
    D = pcd_b200.chamfer_matrix(G.cuda(), R.cuda())
    assert torch.allclose(D.cpu(), O.chamfer_matrix(G, R), rtol=3e-6)
    diag = pcd_b200.chamfer_distance_per_pair(G[:5].cuda(), R.cuda())
    assert torch.allclose(torch.diagonal(D)[:5], diag, rtol=1e-6)
    got = pcd_b200.evaluate_sets(G.cuda(), R.cuda())
    want = O.set_metrics_from_matrices(O.chamfer_matrix(G, R), O.chamfer_matrix(G, G), O.chamfer_matrix(R, R))
    assert same_set_metrics(got, want)


def test_evaluate_sets_tiled_triangle_schedule_on_the_kernels():
    """Several blocks per side (tile 128 on 300 / 260 clouds): the block schedule, the symmetric-triangle shortcut and the
    (value, index) keys against the assembled-matrix definition computed by the oracle."""
    g = torch.Generator().manual_seed(45)
    G = torch.randn(300, 256, 3, generator=g) * (0.2 + 0.8 * torch.rand(300, 1, 3, generator=g))
    R = torch.randn(260, 256, 3, generator=g) * (0.2 + 0.8 * torch.rand(260, 1, 3, generator=g))
    got = pcd_b200.evaluate_sets(G.cuda(), R.cuda(), tile=128)
    Dgr, Dgg, Drr = (pcd_b200.chamfer_matrix(a.cuda(), b.cuda()).cpu() for a, b in ((G, R), (G, G), (R, R)))
    want = O.set_metrics_from_matrices(Dgr, Dgg, Drr)
    assert same_set_metrics(got, want)
    assert torch.equal(Dgg, Dgg.t()) and torch.equal(Drr, Drr.t())       # what the triangle shortcut relies on


@pytest.mark.parametrize("n", [1, 2, 7, 33])
def test_matrix_of_a_set_against_itself_mirrors_the_upper_triangle(n):
    """pcd_chamfer_matrix(G, G) evaluates n (n + 1) / 2 pairs and mirrors them; the values must be those of the full sweep, bit for
    bit (a clone has another address, so it takes the all-pairs path).  Row 0 of the larger sets is degenerate, one has a NaN and
    one a +inf in y (inf - inf makes the reference's scale NaN)."""
    g = torch.Generator().manual_seed(100 + n)
    G = torch.randn(n, 300, 3, generator=g).cuda()
    if n >= 7:
        G[0] = 0.25                     # degenerate cloud -> NaN row and column (metrics.py:19-20)
        G[3, 17, 1] = float("nan")
        G[5, 9, 1] = float("inf")
    full = pcd_b200.chamfer_matrix(G, G.clone())
    tri = pcd_b200.chamfer_matrix(G, G)
    assert tri.shape == (n, n)
    if n >= 7:
        bad = torch.zeros(n, dtype=torch.bool, device="cuda")
        bad[[0, 3, 5]] = True
        assert torch.equal(torch.isnan(full), bad[:, None] | bad[None, :])
    assert torch.equal(torch.isnan(tri), torch.isnan(full))
    assert torch.equal(torch.nan_to_num(tri, nan=-1.0), torch.nan_to_num(full, nan=-1.0))
    assert torch.equal(torch.nan_to_num(tri, nan=-1.0), torch.nan_to_num(tri.t(), nan=-1.0))


@pytest.mark.parametrize("N,M", [(2, 2), (2, 7), (3, 300), (257, 255), (513, 64), (64, 2049), (4500, 4100), (6500, 6400)])
def test_tiny_and_odd_cloud_sizes_vs_exact_oracle(N, M):
    """Point counts that are no multiple of any tile (the kernels pad with far-away sentinels), down to two points per cloud (one
    point is degenerate: NaN, tested above), up to the fused kernel's shared memory (4500 x 4100 takes 137 of its 200 KB) and
    beyond it (6500 x 6400 takes the directional passes): values against the exact oracle, indices bit-exact up to ties, all-pairs
    matrix consistent with the pairs."""
    g = torch.Generator().manual_seed(1000 * N + M)
    x = torch.randn(3, N, 3, generator=g) * torch.rand(3, 1, 3, generator=g)
    y = torch.randn(3, M, 3, generator=g) * torch.rand(3, 1, 3, generator=g) + 0.2
    cd_ref, ixy_ref, iyx_ref = O.chamfer_pairs(x, y)
    cd = pcd_b200.chamfer_distance_per_pair(x.cuda(), y.cuda())
    assert torch.allclose(cd.cpu(), cd_ref, rtol=3e-6)
    cd2, ixy, iyx = pcd_b200._lib.chamfer_pairs(x.cuda(), y.cuda(), 1e3, return_indices=True)
    assert torch.allclose(cd2.cpu(), cd_ref, rtol=3e-6)
    assert float((ixy.cpu().long() != ixy_ref).float().mean()) < 2e-3 and float((iyx.cpu().long() != iyx_ref).float().mean()) < 2e-3
    if N == M or N <= 513:
        yy = y if N == M else torch.randn(2, N, 3, generator=g)
        Dm = pcd_b200.chamfer_matrix(x.cuda(), yy.cuda())
        want = torch.stack([O.chamfer_pairs(x[i:i + 1].expand(yy.shape[0], -1, -1).contiguous(), yy)[0] for i in range(3)])
        assert torch.allclose(Dm.cpu(), want, rtol=3e-6)
