"""GPU parity: VAE3DLarge.encode (implicit-GEMM 3-D convolutions on tcgen05: stride-2 layers, learned 1x1 shortcuts; CUDA-core
encoder.0 and fp32 heads) against the oracle, per layer and end to end."""
import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O
import vae3d_encoder_oracle as E
from conftest import rel_l2

pytestmark = pytest.mark.gpu

# per-layer relative L2 of the activations and of mu / logvar, by precision
TAP_TOL = {"bf16x3": 2e-4, "f16mix": 2e-4, "bf16": 4e-2, "f16": 8e-3}
# (measured on B200 over the six grids below: taps 3e-6..1.1e-4 / mu, logvar 1.2e-4 bf16x3; 9e-8..1.3e-4 / 1.3e-4 f16mix;
#  1.9e-3..7.1e-3 / 7.4e-3 bf16; 1.9e-4..9.2e-4 / 9.0e-4 f16 -- the error grows with depth, encoder.11 / 12 are the largest)
LAT_TOL = TAP_TOL
SEQS = (0, 2, 3, 5, 6, 8, 9, 11, 12)


@pytest.fixture(scope="module")
def esd():
    return E.make_synthetic_vae3d_encoder_checkpoint()


@pytest.fixture(scope="module")
def grids():
    """Shape-like occupancy (the oracle decoder's output on seeded latents, thresholded at 0.4), Bernoulli grids at p = 0.1
    and 0.5, an all-zero and an all-one grid."""
    g = torch.Generator().manual_seed(7)
    shapes = (O.vae3d_decode(O.make_synthetic_vae3d_decoder_checkpoint(), torch.randn(2, 256, generator=g)) > 0.4).float()
    bern = [(torch.rand(1, 1, 32, 32, 32, generator=g) < p).float() for p in (0.1, 0.5)]
    return torch.cat([shapes] + bern + [torch.zeros(1, 1, 32, 32, 32), torch.ones(1, 1, 32, 32, 32)])


@pytest.fixture(scope="module")
def want(esd, grids):
    taps = {}
    mu, logvar = E.vae3d_encode(esd, grids, taps=taps)
    return taps, mu, logvar


def _engine(esd, precision):
    return pcd_b200.Vae3dEncoderEngine(esd, torch.device("cuda", 0), precision)


@pytest.mark.parametrize("precision", ["bf16x3", "f16mix", "bf16", "f16"])
def test_encoder_taps_vs_oracle(esd, grids, want, precision):
    """Every layer of the encoder nn.Sequential against the oracle's activation (localises a wrong tap / shortcut / fold)."""
    eng = _engine(esd, precision)
    taps = want[0]
    errs = {idx: rel_l2(eng.tap(grids.cuda(), idx), taps[idx]) for idx in SEQS}
    print(precision, {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) < TAP_TOL[precision], errs


@pytest.mark.parametrize("precision", ["bf16x3", "f16mix", "bf16", "f16"])
def test_encode_vs_oracle(esd, grids, want, precision):
    mu, logvar = _engine(esd, precision).encode(grids.cuda())
    e_mu, e_lv = rel_l2(mu, want[1]), rel_l2(logvar, want[2])
    print(precision, "mu", f"{e_mu:.2e}", "logvar", f"{e_lv:.2e}")
    assert mu.shape == want[1].shape and logvar.shape == want[2].shape
    assert max(e_mu, e_lv) < LAT_TOL[precision]


@pytest.mark.parametrize("B", [1, 2, 3, 5])
def test_batch_sizes_and_neighbour_independence(esd, grids, want, B):
    eng = _engine(esd, "bf16x3")
    x = grids[:B].cuda()
    mu, logvar = eng.encode(x)
    assert rel_l2(mu, want[1][:B]) < LAT_TOL["bf16x3"] and rel_l2(logvar, want[2][:B]) < LAT_TOL["bf16x3"]
    for i in range(B):                                     # a sample's latent does not depend on its batch neighbours
        m1, l1 = eng.encode(x[i:i + 1])
        assert torch.equal(m1, mu[i:i + 1]) and torch.equal(l1, logvar[i:i + 1])
    rev_mu, _ = eng.encode(x.flip(0))
    assert torch.equal(rev_mu.flip(0), mu)


def _vae(esd):
    vae = pcd_b200.VAE3DLarge()
    sd = O.make_synthetic_vae3d_decoder_checkpoint()
    sd.update(esd)
    vae.load_state_dict({k[4:]: t for k, t in sd.items()}, strict=True)
    return vae.eval().cuda(), sd


def test_module_encode_and_forward_under_seed(esd, grids, want):
    vae, _ = _vae(esd)
    x = grids[:3].cuda()
    mu, logvar = vae.encode(x)
    assert rel_l2(mu, want[1][:3]) < LAT_TOL["bf16x3"]
    torch.manual_seed(11)
    recon, fmu, flv = vae(x)
    assert torch.equal(fmu, mu) and torch.equal(flv, logvar)
    torch.manual_seed(11)
    std = torch.exp(0.5 * logvar)
    z = mu + torch.randn_like(std) * std
    assert torch.equal(recon, vae.decode(z))
    assert recon.shape == (3, 1, 32, 32, 32)
    # dtype / layout of the input do not matter (cast to fp32, made contiguous)
    m2, _ = vae.encode(x.half().transpose(2, 3).contiguous().transpose(2, 3))
    assert torch.equal(m2, mu)


def test_round_trip_through_default_latent_configuration(esd, grids):
    """encode -> LatentDiffusion(vae).sample3(z=mu, start_t=0.01) -> decode -> points, against the oracle encoder feeding the
    same sampler and the oracle decoder."""
    vae, sd = _vae(esd)
    lsd = O.make_synthetic_latent_checkpoint(num_points=256)
    m = pcd_b200.LatentDiffusion(vae)
    m.load_state_dict({k: v for k, v in lsd.items() if k.startswith("model.")}, strict=False)
    m = m.eval().cuda()
    x = grids[:4]
    mu, _ = vae.encode(x.cuda())
    st = torch.tensor([0.01])
    clouds = m.sample3(4, z=mu, start_t=st, num_steps=4, threshold=0.4)
    want_mu, _ = E.vae3d_encode(sd, x)
    z0 = m.sample3(4, z=want_mu.cuda(), start_t=st, num_steps=4, return_latent=True)
    want_vox = O.vae3d_decode(sd, z0.cpu())
    want = O.voxel_tensor_to_point_clouds(want_vox, 0.4)
    near = int(((want_vox - 0.4).abs() < 1e-3).sum())
    for c, w in zip(clouds, want):
        a = {tuple(p) for p in c.cpu().tolist()}
        b = {tuple(p) for p in w.tolist()}
        assert len(a ^ b) <= near, (len(a ^ b), near)


def test_argument_errors(esd):
    eng = _engine(esd, "bf16x3")
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(2, 32, 32, 32, device="cuda"))
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(1, 1, 16, 16, 16, device="cuda"))
    with pytest.raises(pcd_b200.PcdError, match="B must be positive"):
        eng.encode(torch.zeros(0, 1, 32, 32, 32, device="cuda"))
    with pytest.raises(pcd_b200.PcdError):
        eng.encode(torch.zeros(1, 1, 32, 32, 32))                         # host tensor: no CPU fallback
    with pytest.raises(pcd_b200.PcdError, match="seq_index"):
        eng.tap(torch.zeros(1, 1, 32, 32, 32, device="cuda"), 4)
    dec_only = O.make_synthetic_vae3d_decoder_checkpoint()
    dec_only.update({k: v for k, v in esd.items() if k.startswith(("vae.fc_mu", "vae.fc_logvar"))})
    with pytest.raises(pcd_b200.PcdError, match=r"missing: vae\.encoder\."):
        _engine(dec_only, "bf16x3")
    with pytest.raises(pcd_b200.PcdError, match="missing"):
        _engine(O.make_synthetic_vae3d_decoder_checkpoint(), "bf16x3")
    # decoder-only tables keep building decoder handles
    pcd_b200.Vae3dEngine(O.make_synthetic_vae3d_decoder_checkpoint(), torch.device("cuda", 0), "bf16x3").close()
