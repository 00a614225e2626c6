"""GPU: the Sinkhorn EMD kernels (csrc/emd.cu, reference metrics.py:94-158) against a float64 restatement of the reference.

`sinkhorn_f64` below is the reference's recipe with every step in fp64: cube normalisation, direct-difference cdist, ONE cost
maximum over the batch, log(1/n + 1e-10), duals from 0 updated alpha then beta, and the convergence test on both max-abs dual
changes.  (`O.sinkhorn_emd` on double inputs would still keep mu / nu and the first duals in fp32.)

Accuracy rule.  Values are compared at thresh = 0, so both sides run exactly max_iter iterations: a converged dual change of 1e-5
at epsilon = 1e-2 still moves the value by about 1e-3 relative, so an iteration-count mismatch would swamp the comparison.  The
kernel's error against fp64 must be at most 8x the fp32 oracle's (`O.sinkhorn_emd(exact=True)`), plus 2e-6 |fp64|.  Where the
fp64 value is below 1e-30, fp32 underflows: the kernel must return a finite value in [0, 1e-30] there.  Where fp64 overflows to
+inf, the kernel must return +inf.

epsilon > 1.  The reference adds the duals to -C / epsilon without dividing them by epsilon, so each half-step multiplies a uniform
shift of the duals by epsilon.  Below 1 that is a contraction (about epsilon^2 per iteration, which is why most calls stop after a
few iterations); at 1 it is the textbook log-domain Sinkhorn; above 1 the duals diverge, and at epsilon = 10 the value is +inf in
fp64 after one iteration."""
import math

import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O

gpu = pytest.mark.gpu       # every test but the last (a CPU check of the restatement) needs the device


def sinkhorn_f64(x: torch.Tensor, y: torch.Tensor, epsilon: float, thresh: float, max_iter: int):
    """Reference metrics.py:94-158 in fp64 -> (emd[B] per pair, iterations run)."""
    x = O.normalize_to_cube(x.double())
    y = O.normalize_to_cube(y.double())
    C = torch.cdist(x, y, compute_mode="donot_use_mm_for_euclid_dist")
    C = C / C.max()
    lam = 1.0 / epsilon
    B, n, m = C.shape
    log_mu, log_nu = math.log(1.0 / n + 1e-10), math.log(1.0 / m + 1e-10)
    alpha = torch.zeros(B, n, 1, dtype=torch.float64)
    beta = torch.zeros(B, m, 1, dtype=torch.float64)
    iters = 0
    for _ in range(max_iter):
        alpha_prev, beta_prev = alpha, beta
        alpha = epsilon * (log_mu - torch.logsumexp(-lam * C + beta.transpose(1, 2), dim=2, keepdim=True))
        beta = epsilon * (log_nu - torch.logsumexp(-lam * C.transpose(1, 2) + alpha.transpose(1, 2), dim=2, keepdim=True))
        iters += 1
        if (alpha - alpha_prev).abs().max() < thresh and (beta - beta_prev).abs().max() < thresh:
            break
    P = torch.exp(-lam * C + alpha + beta.transpose(1, 2))
    return (P * C).sum(dim=(1, 2)), iters


def _clouds(seed, B, N, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, N, 3, generator=g) * (0.2 + torch.rand(B, 1, 3, generator=g)) + shift


def _pair(N, M, B=3):
    return _clouds(7 * N + M, B, N), _clouds(N + 5 * M + 1, B, M, 0.1)


def assert_f64_rule(got: torch.Tensor, o32: torch.Tensor, want: torch.Tensor):
    """The accuracy rule of the module docstring; returns the kernel / fp32-oracle error ratio of every regular pair."""
    got, o32 = got.cpu().double(), o32.double()
    over = torch.isinf(want)
    assert torch.equal(got[over], want[over]), (got, want)
    tiny = want.abs() < 1e-30
    assert bool(((got[tiny] >= 0) & (got[tiny] <= 1e-30)).all()), (got[tiny], want[tiny])
    reg = ~(over | tiny)
    assert bool(torch.isfinite(got[reg]).all()), got
    err_k, err_o, ref = (got - want).abs()[reg], (o32 - want).abs()[reg], want.abs()[reg]
    ratio = err_k / err_o.clamp_min(1e-300)
    assert bool((err_k <= 8 * err_o + 2e-6 * ref).all()), (
        f"kernel rel err {(err_k / ref).tolist()}, fp32 oracle rel err {(err_o / ref).tolist()}, ratio {ratio.tolist()}")
    return ratio


def check_values(x, y, epsilon, max_iter):
    """thresh = 0: exactly max_iter iterations on both sides; the kernel against fp64 under the accuracy rule."""
    want, it64 = sinkhorn_f64(x, y, epsilon, 0.0, max_iter)
    o32, _ = O.sinkhorn_emd(x, y, epsilon=epsilon, thresh=0.0, max_iter=max_iter, exact=True, per_pair=True)
    got, it = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda(), epsilon, 0.0, max_iter)
    assert it == it64 == max_iter
    return assert_f64_rule(got, o32, want)


# ---- sizes --------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("N,M", [(2, 2), (2, 3), (3, 5), (5, 2),       # the 4-wide target groups padded with -inf in group 0
                                 (257, 1023), (1024, 1024),
                                 (1025, 1025),                           # a second 1024-point target tile holding one point
                                 (255, 2049), (2, 3000), (3000, 2)])
def test_sizes_against_f64(N, M):
    x, y = _pair(N, M)
    check_values(x, y, 1e-2, 30)


@gpu
def test_largest_single_pair_against_f64():
    x, y = _pair(4100, 4100, B=1)
    check_values(x, y, 1e-2, 20)


# ---- epsilon ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("epsilon", [1e-3, 1e-2, 0.1, 1.0])
def test_epsilon_against_f64(epsilon):
    x, y = _pair(512, 480)
    check_values(x, y, epsilon, 30)


@gpu
@pytest.mark.parametrize("max_iter", [0, 1])
def test_epsilon_10_diverges_like_the_reference(max_iter):
    """Without an update the value is finite; one iteration at epsilon = 10 overflows to +inf in fp64, and the kernel follows."""
    x, y = _pair(512, 480)
    want, _ = sinkhorn_f64(x, y, 10.0, 0.0, max_iter)
    assert bool(torch.isfinite(want).all()) == (max_iter == 0)
    check_values(x, y, 10.0, max_iter)


# ---- iteration semantics ------------------------------------------------------------------------------------------------
@gpu
def test_max_iter_0_is_the_plain_kernel_sum():
    """No update: emd = sum_ij exp(-C_ij / eps) C_ij with zero duals, and 0 iterations reported."""
    x, y = _pair(300, 200)
    C = torch.cdist(O.normalize_to_cube(x.double()), O.normalize_to_cube(y.double()), compute_mode="donot_use_mm_for_euclid_dist")
    C = C / C.max()
    plain = (torch.exp(-C / 1e-2) * C).sum(dim=(1, 2))
    want, _ = sinkhorn_f64(x, y, 1e-2, 1e-5, 0)
    assert torch.allclose(want, plain, rtol=1e-14, atol=0)
    check_values(x, y, 1e-2, 0)


@gpu
def test_max_iter_1_and_thresh_bounds():
    x, y = _pair(300, 200)
    check_values(x, y, 1e-2, 1)
    check_values(x, y, 1e-2, 7)                  # thresh = 0: exactly max_iter iterations
    one, it1 = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda(), 1e-2, 0.0, 1)
    inf, it_inf = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda(), 1e-2, float("inf"), 100)
    assert it1 == 1 and it_inf == 1              # every finite change is < inf: one iteration
    assert torch.equal(inf, one)


@gpu
@pytest.mark.parametrize("N,M", [(3, 5), (257, 1023), (1025, 1025), (255, 2049), (2, 3000), (3000, 2)])
@pytest.mark.parametrize("epsilon", [1e-2, 0.3])
def test_default_thresh_iteration_count_ragged(N, M, epsilon):
    """thresh = 1e-5 compares fp32 noise with the threshold: the count agrees with the fp32 oracle and with fp64 within 1."""
    x, y = _pair(N, M, B=2)
    _, it32 = O.sinkhorn_emd(x, y, epsilon=epsilon, thresh=1e-5, max_iter=100, exact=True, per_pair=True)
    _, it64 = sinkhorn_f64(x, y, epsilon, 1e-5, 100)
    _, it = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda(), epsilon, 1e-5, 100)
    assert abs(it - it32) <= 1 and abs(it - it64) <= 1, (it, it32, it64)


# ---- batch coupling -----------------------------------------------------------------------------------------------------
def _coupled_batch():
    """Three pairs that converge at different speeds alone (fp64 counts 3, 5 and 4 at epsilon = 1; 4 together) and whose cost
    maxima differ (pair 2 holds the batch's)."""
    g = torch.Generator().manual_seed(88)
    blob = torch.randn(256, 3, generator=g)
    centres = [torch.randn(4, 3, generator=g) * 3 for _ in range(2)]
    clus = [c[torch.randint(0, 4, (256,), generator=g)] + 0.01 * torch.randn(256, 3, generator=g) for c in centres]
    line = torch.randn(256, 3, generator=g) * torch.tensor([1.0, 0.02, 0.02])
    cube = torch.rand(256, 3, generator=g) * 2 - 1
    return torch.stack([blob, clus[0], line]), torch.stack([blob.clone(), clus[1], cube])


@gpu
def test_batch_converges_together_and_shares_one_cost_maximum():
    x, y = _coupled_batch()
    alone_counts = [sinkhorn_f64(x[i:i + 1], y[i:i + 1], 1.0, 1e-5, 100)[1] for i in range(3)]
    assert len(set(alone_counts)) == 3, alone_counts            # the pairs converge at different speeds alone
    _, it64 = sinkhorn_f64(x, y, 1.0, 1e-5, 100)
    got, it = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda(), 1.0, 1e-5, 100)
    assert abs(it - it64) <= 1, (it, it64)
    # every pair is the fp64 BATCHED value at the batch's count (one cost maximum, one convergence test) ...
    want, _ = sinkhorn_f64(x, y, 1.0, 0.0, it)
    o32, _ = O.sinkhorn_emd(x, y, epsilon=1.0, thresh=0.0, max_iter=it, exact=True, per_pair=True)
    assert_f64_rule(got, o32, want)
    # ... which is not the value of the pair alone (pairs 0 and 1 do not hold the batch maximum)
    alone = torch.cat([sinkhorn_f64(x[i:i + 1], y[i:i + 1], 1.0, 0.0, it)[0] for i in range(3)])
    assert bool(((alone - want).abs()[:2] > 1e-2 * want[:2]).all()), (alone, want)
    # a pair alone is the fp64 value alone
    for i in range(3):
        check_values(x[i:i + 1], y[i:i + 1], 1.0, it)


@gpu
def test_600_small_pairs():
    """B = 600: grid.y is 600 pairs, well past one wave of CTAs; one cost maximum over all of them."""
    x, y = _clouds(600, 600, 64), _clouds(601, 600, 64, 0.1)
    check_values(x, y, 1e-2, 10)


@gpu
def test_deterministic():
    """Fixed-order reductions and an order-free atomicMax: two calls agree bit for bit."""
    x, y = _pair(1025, 1025)
    xc, yc = x.cuda(), y.cuda()
    a, ia = pcd_b200._lib.sinkhorn_emd(xc, yc, 1e-2, 1e-5, 100)
    b, ib = pcd_b200._lib.sinkhorn_emd(xc, yc, 1e-2, 1e-5, 100)
    assert ia == ib and torch.equal(a, b)


# ---- wrapper and C ABI --------------------------------------------------------------------------------------------------
@gpu
def test_argument_errors():
    x, y = _pair(64, 48)
    xc, yc = x.cuda(), y.cuda()
    with pytest.raises(pcd_b200.PcdError, match="must be positive"):
        pcd_b200._lib.sinkhorn_emd(xc[:0], yc[:0])
    with pytest.raises(pcd_b200.PcdError, match="epsilon must be positive"):
        pcd_b200._lib.sinkhorn_emd(xc, yc, 0.0)
    with pytest.raises(pcd_b200.PcdError, match="epsilon must be positive"):
        pcd_b200._lib.sinkhorn_emd(xc, yc, -1e-2)
    with pytest.raises(pcd_b200.PcdError, match="max_iter non-negative"):
        pcd_b200._lib.sinkhorn_emd(xc, yc, 1e-2, 1e-5, -1)
    big = torch.randn(65536, 2, 3, device="cuda")
    with pytest.raises(pcd_b200.PcdError, match="65535"):
        pcd_b200._lib.sinkhorn_emd(big, big)
    with pytest.raises(AssertionError, match="batch sizes"):
        pcd_b200._lib.sinkhorn_emd(xc, yc[:2])


@gpu
def test_float64_and_strided_inputs_and_scaling():
    x, y = _pair(300, 200)
    ref, it = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda())
    got, it2 = pcd_b200._lib.sinkhorn_emd(x.double().cuda(), y.double().cuda())
    assert it2 == it and torch.equal(got, ref)
    xs = torch.empty(3, 3, 300, device="cuda").copy_(x.transpose(1, 2)).transpose(1, 2)        # stride (900, 1, 300)
    ys = torch.empty(3, 400, 3, device="cuda")[:, ::2].copy_(y)                                 # every second point
    assert not xs.is_contiguous() and not ys.is_contiguous()
    got, it2 = pcd_b200._lib.sinkhorn_emd(xs, ys)
    assert it2 == it and torch.equal(got, ref)
    scaled, _ = pcd_b200._lib.sinkhorn_emd(x.cuda(), y.cuda(), scaling=7.0)
    assert torch.equal(scaled, ref * 7.0)
    mean = pcd_b200.earth_mover_distance_gpu(x.cuda(), y.cuda())
    assert torch.equal(mean, ref.mean())
    assert torch.equal(pcd_b200.earth_mover_distance_gpu(x.cuda(), y.cuda(), scaling_factor=3.5), ref.mean() * 3.5)


def test_f64_restatement_tracks_the_oracle():
    """CPU: the fp64 restatement and the fp32 oracle agree to fp32 noise, with the same iteration count."""
    x, y = _pair(96, 80)
    for epsilon in (1e-2, 0.3, 1.0):
        want, it64 = sinkhorn_f64(x, y, epsilon, 1e-5, 100)
        o32, it32 = O.sinkhorn_emd(x, y, epsilon=epsilon, thresh=1e-5, max_iter=100, exact=True, per_pair=True)
        assert it64 == it32 and torch.allclose(o32.double(), want, rtol=2e-5, atol=0), (epsilon, o32, want)

