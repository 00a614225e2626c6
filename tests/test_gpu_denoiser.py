"""GPU: the denoiser forward through the C ABI against the oracle / reference golden vectors.

Tolerances (relative L2 on eps_hat, per forward):
  fp32 mode : 1e-5  (north_star's fp32 bound; measured noise floor of the fp32 oracle itself is
              1.4e-6 between batch sizes, SURVEY appendix B)
  bf16x3    : 1e-3  (north_star's bf16 bound) -- hi+lo bf16 planes, 3 MMAs per k-step, fp32 accumulate
  f16mix    : 1e-3  (north_star's bound again) -- fp16 hi+lo planes with 3 MMAs everywhere except
              global_feat.0/.3 (67 % of the FLOPs), which run ONE fp16 pass: ~1.7x the cost of a pass
  f16 mode  : 6e-3  -- one fp16 pass per layer: the speed of bf16 mode with 3 more mantissa bits
              (measured ~2.6e-3)
  bf16 mode : 3e-2  -- north_star asks 1e-3, but SURVEY H2 measured that NO single-pass bf16
              pipeline can meet it on this 28-layer net (bf16 W x bf16 A with fp32 accumulate
              gives 1.2e-2 even in pure torch emulation).  We assert 3e-2 here and, separately,
              that our kernel is as accurate as a torch emulation of the same bf16 pipeline.
"""
import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O
from conftest import rel_l2

pytestmark = pytest.mark.gpu

TOL = {"fp32": 1e-5, "bf16": 3e-2, "bf16x3": 1e-3, "f16": 6e-3, "f16mix": 1e-3}
ALL = ["fp32", "bf16", "bf16x3", "f16", "f16mix"]   # bf16x3 = north_star's 1e-3 bound, met with split-bf16 operands


def _model(sd, precision, n=256):
    m = pcd_b200.PointCloudDiffusion(n, precision=precision)
    m.load_state_dict(sd, strict=True)
    return m.eval().cuda()


@pytest.mark.parametrize("precision", ALL)
def test_forward_vs_reference_golden(golden, sd33, precision):
    m = _model(sd33, precision)
    for tag in ("fwd", "fwd2"):     # fwd2: B=3, N=200 (ragged, not a multiple of 128)
        x, t = golden[f"a33.{tag}.x"].cuda(), golden[f"a33.{tag}.t"].cuda()
        eps = m.model(x, t)
        assert eps.shape == x.shape and eps.is_cuda
        assert torch.isfinite(eps).all()
        assert rel_l2(eps, golden[f"a33.{tag}.eps"]) < TOL[precision]


@pytest.mark.parametrize("precision", ALL)
def test_forward_taps_vs_oracle(sd33, precision, monkeypatch):
    """Layer-by-layer check of the intermediate activations (localises a bug to a block)."""
    monkeypatch.setenv("PCD_TAPS", "1")
    m = _model(sd33, precision)
    g = torch.Generator().manual_seed(21)
    B, N = 2, 384
    x, t = torch.randn(B, N, 3, generator=g), torch.tensor([0.25, 0.8])
    taps = {}
    ref = O.denoiser_forward(sd33, x, t, taps=taps)
    eps = m.model(x.cuda(), t.cuda())
    eng = m.model.engine()
    tol = {"fp32": 5e-6, "bf16": 2e-2, "bf16x3": 2e-4, "f16": 4e-3, "f16mix": 1e-3}[precision]
    assert rel_l2(eng.tap("temb", (B, 256)), taps["temb"]) < 5e-6
    for name, C in (("x1", 128), ("x2", 256), ("x3", 512), ("x4", 1024), ("d4", 512), ("d1", 64)):
        got = eng.tap(name, (B, N, C))             # N is a multiple of 128 here: no padding rows
        want = taps[name].transpose(1, 2)          # oracle is channel-major [B,C,N]
        assert rel_l2(got, want) < tol, name
    assert rel_l2(eng.tap("g", (B, 4096)), taps["g"]) < tol
    assert rel_l2(eps, ref) < TOL[precision]


def test_bf16_kernel_is_as_accurate_as_a_torch_bf16_emulation(sd33):
    """Our bf16 result must be no worse than 1.5x the error of the same pipeline emulated in torch
    (bf16-rounded weights and activations, fp32 accumulate)."""
    g = torch.Generator().manual_seed(22)
    x, t = torch.randn(2, 256, 3, generator=g), torch.tensor([0.6, 0.05])
    ref = O.denoiser_forward(sd33, x, t)

    def q(v):
        return v.bfloat16().float()
    sdq = {k: (q(v) if k.endswith("weight") and v.dim() >= 2 else v) for k, v in sd33.items()}
    emu_err = rel_l2(O.denoiser_forward(sdq, x, t), ref)    # weight rounding only: a lower bound
    m = _model(sd33, "bf16")
    got_err = rel_l2(m.model(x.cuda(), t.cuda()), ref)
    assert got_err < max(3.0 * emu_err, 1e-2), (got_err, emu_err)


@pytest.mark.parametrize("precision", ALL)
def test_point_permutation_equivariance(sd33, precision):
    m = _model(sd33, precision)
    g = torch.Generator().manual_seed(23)
    x, t = torch.randn(2, 256, 3, generator=g).cuda(), torch.tensor([0.4, 0.9]).cuda()
    perm = torch.randperm(256, generator=g).cuda()
    a = m.model(x, t)[:, perm]
    b = m.model(x[:, perm].contiguous(), t)
    # per-point layers are row-independent and max is order independent: identical up to the
    # atomicMax order (exact) -> bitwise equal
    assert torch.equal(a, b)


@pytest.mark.parametrize("precision", ALL)
def test_batch_shard_invariance(sd33, precision):
    m = _model(sd33, precision)
    g = torch.Generator().manual_seed(24)
    x, t = torch.randn(4, 128, 3, generator=g).cuda(), torch.tensor([0.4, 0.9, 0.1, 1.0]).cuda()
    full = m.model(x, t)
    halves = torch.cat([m.model(x[:2].contiguous(), t[:2].contiguous()), m.model(x[2:].contiguous(), t[2:].contiguous())])
    assert torch.equal(full, halves)


def test_engine_rebuilds_when_weights_change(sd33):
    m = _model(sd33, "fp32", 128)
    x, t = torch.randn(1, 128, 3).cuda(), torch.tensor([0.5]).cuda()
    a = m.model(x, t)
    with torch.no_grad():
        m.model.output[3].weight.mul_(2.0)
        m.model.output[3].bias.mul_(2.0)
    b = m.model(x, t)
    assert torch.allclose(b, 2 * a, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("precision", ["bf16", "f16mix", "bf16x3"])
@pytest.mark.parametrize("B,N", [(3, 128), (1, 100), (5, 300)])
def test_odd_tile_counts_take_the_single_cta_path(sd33, precision, B, N):
    """B*ceil(N/128) odd -> no CTA pairs (one CTA per tile, cta_group::1, 128-point max-pool tiles): same answers."""
    g = torch.Generator().manual_seed(25)
    x, t = torch.randn(B, N, 3, generator=g), torch.rand(B, generator=g)
    ref = O.denoiser_forward(sd33, x, t)
    eps = _model(sd33, precision).model(x.cuda(), t.cuda())
    assert rel_l2(eps, ref) < TOL[precision]


def test_single_cta_and_pair_schemes_agree_bitwise(sd33):
    """B = 3, N = 128 is three 128-row blocks: every per-point layer runs one CTA per tile (cta_group::1, no multicast).  B = 4
    pairs its row blocks: TMA multicast with per-CTA MMAs on the K < 1024 layers, the pair MMA (cta_group::2) on the K >= 1024
    layers.  All three schemes accumulate in the same order, so the first three clouds get identical bits."""
    g = torch.Generator().manual_seed(26)
    x, t = torch.randn(4, 128, 3, generator=g).cuda(), torch.tensor([0.3, 0.7, 0.1, 0.9]).cuda()
    m = _model(sd33, "bf16", 128)
    four = m.model(x, t)
    three = m.model(x[:3].contiguous(), t[:3].contiguous())
    assert torch.equal(three, four[:3])


def test_plan_cache_keeps_only_recent_shapes(sd33, monkeypatch):
    """A plan owns the workspace of one (B, N) shape; the handle keeps the PCD_MAX_PLANS most recently used ones and frees the
    rest, so a caller sweeping batch sizes does not accumulate workspaces; results do not depend on cache hits or evictions."""
    monkeypatch.setenv("PCD_MAX_PLANS", "2")
    m = _model(sd33, "bf16", 2048)
    g = torch.Generator().manual_seed(26)
    xs = {B: torch.randn(B, 2048, 3, generator=g).cuda() for B in (2, 16, 32, 48)}
    ts = {B: torch.full((B,), 0.5).cuda() for B in xs}
    first = m.model(xs[2], ts[2]).clone()
    torch.cuda.synchronize()
    free = []
    for rnd in range(2):
        for B in (16, 32, 48):                              # ~0.35 / 0.7 / 1.05 GB of workspace each
            m.model(xs[B], ts[B])
            torch.cuda.synchronize()
            free.append(torch.cuda.mem_get_info()[0])
    assert torch.equal(m.model(xs[2], ts[2]), first)        # evicted and rebuilt: same bits
    # the second sweep re-creates evicted plans instead of stacking new ones: free memory stays within one large plan of the first sweep
    assert min(free[3:]) > min(free[:3]) - 1.3e9


@pytest.mark.parametrize("T", [64, 129, 512])
def test_other_time_widths_vs_oracle(T):
    """dim == time_dim != 256 (reference constructor kwargs, diffusion.py:15-28): only the time MLP and the temb columns of
    enc1.conv1 depend on it.  fp32 mode within the 1e-5 bound, f16mix within 1e-3; the DDIM loop runs on the same handle."""
    sd = O.make_synthetic_checkpoint(seed=24, alpha=1.0 / 33.0, dim=T, time_dim=T)
    g = torch.Generator().manual_seed(15)
    x, t = torch.randn(3, 200, 3, generator=g), torch.tensor([0.05, 0.5, 1.0])
    ref = O.denoiser_forward(sd, x, t, time_dim=T)
    for precision, bound in (("fp32", 1e-5), ("f16mix", 1e-3)):
        m = pcd_b200.PointCloudDiffusion(200, dim=T, time_dim=T, precision=precision)
        m.load_state_dict(sd, strict=True)
        m = m.eval().cuda()
        assert rel_l2(m.model(x.cuda(), t.cuda()), ref) < bound, (T, precision)
        if precision == "fp32":
            assert rel_l2(m.sample(3, 200, num_steps=4, x_T=x), O.ddim_sample(sd, x, 4)) < 2e-4


@pytest.mark.parametrize("B,N", [(1, 384), (1, 2048), (3, 1000)])
def test_f16mix_plans_with_and_without_the_fp8_pass(sd33, B, N):
    """f16mix runs the tensor-bound split layers with an fp8 correction pass on CTA pairs; a plan whose 128-row blocks do not pair
    up (B * ceil(N / 128) odd: 3 blocks here) falls back to three fp16 passes on the weights' fp16 residual plane, and the tensors
    between those layers carry fp16 residuals instead of byte planes.  Both plans must sit inside the 1e-3 bound."""
    g = torch.Generator().manual_seed(16)
    x, t = torch.randn(B, N, 3, generator=g), torch.rand(B, generator=g)
    ref = O.denoiser_forward(sd33, x, t)
    m = pcd_b200.PointCloudDiffusion(N, precision="f16mix")
    m.load_state_dict(sd33, strict=True)
    m = m.eval().cuda()
    assert rel_l2(m.model(x.cuda(), t.cuda()), ref) < 1e-3


def test_fp16_planes_saturate_on_out_of_range_activations(sd33):
    """fp16 tops out at 65504; coordinates 2e4 x larger than a diffusion state drive the early activations past it.  The fp16 modes
    clamp (pcd_types.h: a finite, wrong-by-saturation value instead of inf -> NaN through the next layer's BN fold); the bf16 planes
    have fp32's exponent range, so `bf16x3` still matches the reference's fp32 result -- the mode to pick for such a checkpoint."""
    g = torch.Generator().manual_seed(8)
    x = torch.randn(2, 256, 3, generator=g) * 2.0e4
    t = torch.tensor([0.2, 0.8])
    ref = O.denoiser_forward(sd33, x, t)
    assert float(ref.abs().max()) > 1e3 and bool(torch.isfinite(ref).all())
    for precision in ("f16mix", "f16", "bf16x3", "bf16"):
        m = pcd_b200.PointCloudDiffusion(256, precision=precision)
        m.load_state_dict(sd33, strict=True)
        out = m.eval().cuda().model(x.cuda(), t.cuda())
        assert bool(torch.isfinite(out).all()), precision
        if precision == "bf16x3":
            assert rel_l2(out, ref) < 1e-3              # measured 7.3e-5
        if precision == "bf16":
            assert rel_l2(out, ref) < 6e-2              # measured 3.2e-2
        if precision in ("f16mix", "f16"):
            assert rel_l2(out, ref) > 0.1               # clamped (measured ~1.0): the diagnostic below must flag it
            assert m.model.precision_gap(x.cuda(), t.cuda()) > 0.1
    m = pcd_b200.PointCloudDiffusion(256, precision="f16mix")          # in range: the gap is the mode's own error
    m.load_state_dict(sd33, strict=True)
    assert m.eval().cuda().model.precision_gap((x / 2.0e4).cuda(), t.cuda()) < 2e-3
