"""GPU: SimplePointNetVAE.encode (a PointNet trunk on the tcgen05 per-point GEMMs with the max-pool fused into encoder.3.conv3's
epilogue; CUDA-core first layer and fp32 heads) against the oracle per layer and end to end, and the exactness properties of a
PointNet: batch independence, point-permutation invariance, padded rows never reaching the max, and NaN for non-finite clouds."""
import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O
import point_vae_encoder_oracle as P
from conftest import rel_l2

pytestmark = pytest.mark.gpu

# per-layer relative L2 of the activations and of mu / logvar, by precision (the voxel encoder's bounds)
TOL = {"bf16x3": 2e-4, "f16mix": 2e-4, "bf16": 4e-2, "f16": 8e-3}
# (measured on B200, worst over the clouds below: taps 3.5e-6..2.0e-5 / mu, logvar 1.7e-5 bf16x3; 9e-8..8.0e-6 / 8.0e-6 f16mix;
#  1.9e-3..1.3e-2 / 1.2e-2 bf16; 2.2e-4..1.7e-3 / 1.6e-3 f16 -- the error grows with depth, encoder.3 and the heads are the largest)
PRECISIONS = ["bf16x3", "f16mix", "bf16", "f16"]
NP = 512          # points of the decoder that makes the shape-like clouds and of the round-trip VAE


@pytest.fixture(scope="module")
def esd():
    return P.make_synthetic_point_vae_encoder_checkpoint()


@pytest.fixture(scope="module")
def lsd():
    return O.make_synthetic_latent_checkpoint(num_points=NP)


@pytest.fixture(scope="module")
def clouds(lsd):
    """name -> [B, N, 3]: Gaussian clouds, cube-normalised decoder outputs on seeded latents, a cloud whose points are all
    equal, and Gaussian clouds of N = 1, 100, 128, 129 and 2500 points (2048 above)."""
    g = torch.Generator().manual_seed(7)
    shapes = O.normalize_to_cube(O.vae_decode(lsd, torch.randn(2, 256, generator=g), NP))
    out = {"gauss2048": torch.randn(2, 2048, 3, generator=g), "shape512": shapes,
           "degenerate300": torch.randn(1, 1, 3, generator=g).expand(1, 300, 3).contiguous()}
    for n in (1, 100, 128, 129, 2500):
        out[f"gauss{n}"] = torch.randn(2, n, 3, generator=g)
    return out


def _engine(esd, precision="bf16x3"):
    return pcd_b200.PointEncoderEngine(esd, torch.device("cuda", 0), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_taps_and_latents_vs_oracle(esd, clouds, precision):
    """Every conv (after BatchNorm + ReLU, valid points), the pooled feature, encoder.7 and mu / logvar against the oracle."""
    eng = _engine(esd, precision)
    worst = {}
    for name, x in clouds.items():
        taps = {}
        want_mu, want_lv = P.point_vae_encode(esd, x, taps=taps)
        for i in range(14):
            got = eng.tap(x.cuda(), i)
            assert got.shape == taps[i].shape, (name, i)
            worst[i] = max(worst.get(i, 0.0), rel_l2(got, taps[i]))
        mu, logvar = eng.encode(x.cuda())
        worst["mu"] = max(worst.get("mu", 0.0), rel_l2(mu, want_mu))
        worst["logvar"] = max(worst.get("logvar", 0.0), rel_l2(logvar, want_lv))
    print(precision, {k: f"{v:.2e}" for k, v in worst.items()})
    assert max(worst.values()) < TOL[precision], worst


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
@pytest.mark.parametrize("N", [100, 300])
def test_batch_independence(esd, precision, N):
    """A cloud's latent equals the same cloud encoded alone, for batches whose row-block count is odd and even (CTA pairs or
    not, 128- or 256-column tiles), and a reversed batch gives reversed outputs."""
    eng = _engine(esd, precision)
    x = torch.randn(5, N, 3, generator=torch.Generator().manual_seed(N)).cuda()
    alone = [eng.encode(x[i:i + 1]) for i in range(5)]
    for B in (1, 2, 3, 5):
        mu, logvar = eng.encode(x[:B])
        for i in range(B):
            assert torch.equal(mu[i:i + 1], alone[i][0]) and torch.equal(logvar[i:i + 1], alone[i][1]), (B, i)
        rmu, rlv = eng.encode(x[:B].flip(0))
        assert torch.equal(rmu.flip(0), mu) and torch.equal(rlv.flip(0), logvar)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_point_permutation_and_padding(esd, precision):
    """PointNet invariance is exact: rows are independent and max is exact.  Appending a copy of an existing point (N crosses
    128 -> 129, a second row block per cloud) changes nothing, so padded rows never reach the max."""
    eng = _engine(esd, precision)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 128, 3, generator=g)
    mu, logvar = eng.encode(x.cuda())
    perm = torch.randperm(128, generator=g)
    pmu, plv = eng.encode(x[:, perm].cuda())
    assert torch.equal(pmu, mu) and torch.equal(plv, logvar)
    x129 = torch.cat([x, x[:, 17:18]], dim=1)
    amu, alv = eng.encode(x129.cuda())
    assert torch.equal(amu, mu) and torch.equal(alv, logvar)


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), float("-inf")])
def test_non_finite_clouds(esd, bad):
    """A NaN coordinate makes every mu / logvar entry of its cloud NaN, as in the reference; an infinite one gives what the
    oracle gives on this checkpoint (all NaN: +-inf times weights of both signs).  The finite neighbours in the same batch are
    bit-identical to encoding them alone."""
    eng = _engine(esd)
    x = torch.randn(3, 200, 3, generator=torch.Generator().manual_seed(4))
    x[1, 57, 2] = bad
    want_mu, want_lv = P.point_vae_encode(esd, x[1:2])
    assert torch.isnan(want_mu).all() and torch.isnan(want_lv).all()
    mu, logvar = eng.encode(x.cuda())
    assert torch.isnan(mu[1]).all() and torch.isnan(logvar[1]).all()
    for i in (0, 2):
        m1, l1 = eng.encode(x[i:i + 1].cuda())
        assert torch.equal(mu[i:i + 1], m1) and torch.equal(logvar[i:i + 1], l1)


def _vae(esd, lsd):
    vae = pcd_b200.SimplePointNetVAE(NP)
    sd = {k: v for k, v in lsd.items() if k.startswith("vae.")}
    sd.update(esd)
    vae.load_state_dict({k[4:]: t for k, t in sd.items()}, strict=True)
    return vae.eval().cuda(), sd


def test_module_encode_forward_and_inputs(esd, lsd, clouds):
    vae, sd = _vae(esd, lsd)
    x = clouds["shape512"].cuda()
    mu, logvar = vae.encode(x)
    e_mu, e_lv = _engine(esd).encode(x)
    assert torch.equal(mu, e_mu) and torch.equal(logvar, e_lv)
    torch.manual_seed(11)
    recon, fmu, flv = vae(x)
    assert torch.equal(fmu, mu) and torch.equal(flv, logvar)
    torch.manual_seed(11)
    std = torch.exp(0.5 * logvar)
    assert torch.equal(recon, vae.decode(mu + torch.randn_like(std) * std))
    assert recon.shape == (2, NP, 3)
    # dtype / layout of the input do not matter (cast to fp32, made contiguous)
    xh = x.half()
    assert torch.equal(vae.encode(xh)[0], vae.encode(xh.float())[0])
    assert torch.equal(vae.encode(x.transpose(0, 1).contiguous().transpose(0, 1))[0], mu)
    # a train-mode module still encodes with the running statistics (eval-mode BatchNorm)
    vae.train()
    assert torch.equal(vae.encode(x)[0], mu)


def test_round_trip_through_point_latent_configuration(esd, lsd, clouds):
    """LatentDiffusion(SimplePointNetVAE, is_voxel_based=False).sample3(z=vae.encode(x)[0], start_t=0.01) against the oracle
    encoder's mu fed to the same sampler and the oracle decoder: the encoder's error (2e-5 in bf16x3) passes through four
    DDIM steps and the decoder (measured on B200: 1.9e-5 relative L2)."""
    vae, sd = _vae(esd, lsd)
    m = pcd_b200.LatentDiffusion(vae, is_voxel_based=False)
    m.load_state_dict({k: v for k, v in lsd.items() if k.startswith("model.")}, strict=False)
    m = m.eval().cuda()
    x = clouds["shape512"]
    st = torch.tensor([0.01])
    got = m.sample3(2, z=vae.encode(x.cuda())[0], start_t=st, num_steps=4)
    want_mu, _ = P.point_vae_encode(esd, x)
    z0 = m.sample3(2, z=want_mu.cuda(), start_t=st, num_steps=4, return_latent=True)
    want = O.vae_decode(sd, z0.cpu(), NP)
    err = rel_l2(got, want)
    print("round trip rel L2", f"{err:.2e}")
    assert got.shape == (2, NP, 3) and err < 2e-4


def test_argument_errors(esd, lsd):
    eng = _engine(esd)
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(2, 10, device="cuda"))
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(2, 10, 4, device="cuda"))
    with pytest.raises(pcd_b200.PcdError, match="B and N must be positive"):
        eng.encode(torch.zeros(0, 10, 3, device="cuda"))
    with pytest.raises(pcd_b200.PcdError, match="B and N must be positive"):
        eng.encode(torch.zeros(2, 0, 3, device="cuda"))
    with pytest.raises(pcd_b200.PcdError, match="CUDA tensor"):
        eng.encode(torch.zeros(1, 10, 3))                               # host tensor: no CPU fallback
    with pytest.raises(pcd_b200.PcdError, match="index"):
        eng.tap(torch.zeros(1, 10, 3, device="cuda"), 14)
    heads_only = {k: v for k, v in esd.items() if k.startswith(("vae.fc_mu", "vae.fc_logvar"))}
    with pytest.raises(pcd_b200.PcdError, match=r"missing: vae\.encoder\.0\.conv1\.weight"):
        _engine(heads_only)
    with pytest.raises(pcd_b200.PcdError, match="hidden_dim = 512"):
        _engine(P.make_synthetic_point_vae_encoder_checkpoint(hidden_dim=256))
    # decoder-only tables still build a LatentEngine and decode as before
    dec_only = {k: v for k, v in lsd.items() if k.startswith("vae.")}
    le = pcd_b200.latent.LatentEngine(dec_only, NP, torch.device("cuda", 0))
    z = torch.randn(3, 256, generator=torch.Generator().manual_seed(1))
    assert rel_l2(le.decode(z.cuda()), O.vae_decode(lsd, z, NP)) < 2e-5
    le.close()
