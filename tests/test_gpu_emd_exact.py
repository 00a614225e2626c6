"""GPU: exact EMD (reference metrics.py:49-92, `earth_mover_distance_cpu`) through the auction kernel against the known answer
and SciPy's linear_sum_assignment (tests/exact_emd_scipy.py).

Tolerance: |gpu - scipy| <= 2e-6 * scipy + 1e-6 per pair.  The kernel's matching is optimal for distances quantised to 2^-22, which
moves the matched sum by at most n / 2^22 absolute; the rest is fp32 distance error."""
import pytest
import torch

import exact_emd_scipy as S
import pcd_b200
from oracle import pointdiff_oracle as O

pytestmark = pytest.mark.gpu
KNOWN = 44.30706787109375


def _clouds(seed, B, N, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, N, 3, generator=g) * (0.2 + torch.rand(B, 1, 3, generator=g)) + shift


def _check_against_scipy(x, y):
    got, assign = pcd_b200._lib.emd_exact(x.cuda(), y.cuda(), return_assignment=True)
    got, assign = got.cpu().double(), assign.cpu().long()
    want = S.exact_emd(x, y, per_pair=True)
    assert torch.all((got - want).abs() <= 2e-6 * want + 1e-6), (got, want)
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    xn, yn = O.normalize_to_cube(x).double(), O.normalize_to_cube(y).double()
    for b in range(B):
        a = assign[b]
        if N <= M:
            assert bool((a >= 0).all())
        else:
            assert int((a >= 0).sum()) == M
        m = a[a >= 0]
        assert m.unique().numel() == m.numel() and int(m.max()) < M
        rows = torch.nonzero(a >= 0).squeeze(1)
        cost = float((xn[b, rows] - yn[b, m]).norm(dim=1).sum()) / 3          # fp64 cost of the returned assignment
        assert abs(cost - float(got[b])) <= 1e-6 * cost + 1e-7, (b, cost, float(got[b]))
    return got, assign


def test_known_answer_units_inputs(golden):
    x, y = golden["cd.units.x"].cuda(), golden["cd.units.y"].cuda()
    emd = pcd_b200.earth_mover_distance_exact(x, y)
    assert emd.dim() == 0 and emd.is_cuda and emd.dtype == torch.float32
    assert abs(float(emd) - KNOWN) <= 2e-6 * KNOWN
    emd2 = pcd_b200.earth_mover_distance_exact(x[0], y[0])          # 2-D promotion
    assert torch.equal(emd2, emd)


@pytest.mark.parametrize("n", [64, 512, 2048, 4096])
def test_optimal_against_scipy_square(n):
    _check_against_scipy(_clouds(n, 2, n), _clouds(n + 1, 2, n, 0.1))


@pytest.mark.parametrize("N,M", [(994, 948), (948, 994), (2048, 1500), (2, 300), (300, 2), (2, 2)])
def test_optimal_against_scipy_ragged(N, M):
    _check_against_scipy(_clouds(N * 7 + M, 2, N), _clouds(N + 3 * M, 2, M, 0.2))


def test_ties_duplicated_points():
    g = torch.Generator().manual_seed(9)
    base_x, base_y = torch.randn(2, 40, 3, generator=g), torch.randn(2, 30, 3, generator=g)
    x = base_x[:, torch.randint(0, 40, (512,), generator=g)]
    y = base_y[:, torch.randint(0, 30, (400,), generator=g)]
    _check_against_scipy(x, y)
    _check_against_scipy(y, x)
    _check_against_scipy(x, x[:, torch.randperm(512, generator=g)])


def test_exact_zeros_and_inverse_permutation():
    x = _clouds(21, 3, 1024)
    g = torch.Generator().manual_seed(22)
    perm = torch.randperm(1024, generator=g)
    emd, assign = pcd_b200._lib.emd_exact(x.cuda(), x.cuda(), return_assignment=True)
    assert torch.equal(emd.cpu(), torch.zeros(3)) and torch.equal(assign.cpu().long(), torch.arange(1024).expand(3, -1))
    emd, assign = pcd_b200._lib.emd_exact(x.cuda(), x[:, perm].cuda(), return_assignment=True)
    assert torch.equal(emd.cpu(), torch.zeros(3))
    assert torch.equal(assign.cpu().long(), torch.argsort(perm).expand(3, -1))


def test_deterministic_and_batch_independent():
    x, y = _clouds(31, 37, 700), _clouds(32, 37, 650, 0.05)
    a1, s1 = pcd_b200._lib.emd_exact(x.cuda(), y.cuda(), return_assignment=True)
    a2, s2 = pcd_b200._lib.emd_exact(x.cuda(), y.cuda(), return_assignment=True)
    assert torch.equal(a1, a2) and torch.equal(s1, s2)
    for k in (0, 17, 36):
        ak, sk = pcd_b200._lib.emd_exact(x[k:k + 1].cuda(), y[k:k + 1].cuda(), return_assignment=True)
        assert torch.equal(ak[0], a1[k]) and torch.equal(sk[0], s1[k])


def test_degenerate_cloud_is_nan_and_size_limit():
    x, y = _clouds(41, 3, 256), _clouds(42, 3, 200)
    x[1] = 0.5                                                         # all points equal: normalize_to_cube divides by 0
    emd, assign = pcd_b200._lib.emd_exact(x.cuda(), y.cuda(), return_assignment=True)
    emd, assign = emd.cpu(), assign.cpu()
    assert torch.isnan(emd[1]) and bool((assign[1] == -1).all())
    assert torch.isfinite(emd[[0, 2]]).all()
    want = S.exact_emd(x[[0, 2]], y[[0, 2]], per_pair=True)
    assert torch.all((emd[[0, 2]].double() - want).abs() <= 2e-6 * want + 1e-6)
    # a one-point cloud normalises to 0 / 0 as well
    emd, assign = pcd_b200._lib.emd_exact(y[:, :1].cuda(), x.cuda(), return_assignment=True)
    assert torch.isnan(emd.cpu()).all() and bool((assign == -1).all())
    assert torch.isnan(pcd_b200._lib.emd_exact(y.cuda(), y[:, :1].cuda()).cpu()).all()
    with pytest.raises(pcd_b200.PcdError, match="4096"):
        pcd_b200._lib.emd_exact(torch.randn(1, 4097, 3, device="cuda"), torch.randn(1, 64, 3, device="cuda"))
    with pytest.raises(pcd_b200.PcdError, match="4096"):
        pcd_b200.earth_mover_distance_exact(torch.randn(64, 3, device="cuda"), torch.randn(4097, 3, device="cuda"))


def test_compute_metrics_hook():
    x, y = _clouds(51, 4, 512).cuda(), _clouds(52, 4, 480, 0.1).cuda()
    cd, emd, recon = pcd_b200.compute_metrics(x, y, emd_fn=pcd_b200.earth_mover_distance_exact)
    assert all(isinstance(v, torch.Tensor) and v.dim() == 0 for v in (cd, emd, recon))
    assert torch.equal(emd, pcd_b200.earth_mover_distance_exact(x, y))
    assert abs(float(emd) - float(S.exact_emd(x.cpu(), y.cpu()))) <= 2e-6 * float(emd) + 1e-6


def test_emd_matrix_and_evaluate_sets():
    G, R = _clouds(61, 24, 256), _clouds(62, 20, 256, 0.1)
    Gc, Rc = G.cuda(), R.cuda()
    D = pcd_b200.emd_matrix(Gc[:5], Rc[:4]).cpu()
    loop = torch.stack([torch.stack([pcd_b200.earth_mover_distance_exact(Gc[i], Rc[j]) for j in range(4)]) for i in range(5)]).cpu()
    assert torch.equal(D, loop)
    Dgg = pcd_b200.emd_matrix(Gc, Gc)
    assert torch.equal(Dgg, Dgg.t()) and torch.equal(torch.diagonal(Dgg).cpu(), torch.zeros(24))
    want = pcd_b200.set_metrics_from_matrices(pcd_b200.emd_matrix(Gc, Rc), Dgg, pcd_b200.emd_matrix(Rc, Rc))
    for tile in (None, 7):
        got = pcd_b200.evaluate_sets(Gc, Rc, metric="emd", tile=tile)
        assert got["cov_emd"] == want["cov_cd"] and got["1nna_emd"] == pytest.approx(want["1nna_cd"], abs=1e-6)
        assert got["mmd_emd"] == pytest.approx(want["mmd_cd"], rel=1e-6)
