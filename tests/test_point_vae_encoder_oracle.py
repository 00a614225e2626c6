"""CPU: the point-VAE encoder oracle (SimplePointNetVAE.encode) -- the state_dict layout, the no-CPU-fallback rule, the
reparameterisation draw, checkpoint loading with a precision override and, where the reference tree is mounted, the
reference's own encode / forward."""
import pytest
import torch

import pcd_b200
from oracle import pointdiff_oracle as O
from oracle import ref_shim
import point_vae_encoder_oracle as P

NP = 256


def _full_checkpoint():
    """Encoder + decoder of SimplePointNetVAE(NP), without the `vae.` prefix."""
    sd = {k: v for k, v in O.make_synthetic_latent_checkpoint(num_points=NP).items() if k.startswith("vae.")}
    sd.update(P.make_synthetic_point_vae_encoder_checkpoint())
    return {k[4:]: t for k, t in sd.items()}


def test_encoder_spec_matches_container_and_full_checkpoint_loads_strictly():
    v = pcd_b200.SimplePointNetVAE(NP)
    sd = v.state_dict()
    spec = P.point_vae_encoder_state_dict_spec(prefix="vae")
    for k, shape, _ in spec:
        assert tuple(sd[k[4:]].shape) == tuple(shape), k
    enc_keys = {k for k in sd if k.startswith(("encoder.", "fc_mu.", "fc_logvar."))}
    assert enc_keys == {k[4:] for k, _, _ in spec}
    v.load_state_dict(_full_checkpoint(), strict=True)


def test_encode_on_cpu_raises():
    v = pcd_b200.SimplePointNetVAE(NP)
    v.load_state_dict(_full_checkpoint(), strict=True)
    x = torch.zeros(1, 64, 3)
    with pytest.raises(pcd_b200.PcdError):                # no CPU fallback
        v.encode(x)
    with pytest.raises(pcd_b200.PcdError):
        v(x)


def test_reparameterize_draws_like_the_reference():
    mu, logvar = torch.randn(3, 8), torch.randn(3, 8)
    torch.manual_seed(5)
    got = pcd_b200.SimplePointNetVAE.reparameterize(mu, logvar)
    torch.manual_seed(5)
    std = torch.exp(0.5 * logvar)
    assert torch.equal(got, mu + torch.randn_like(std) * std)


def test_load_from_checkpoint_with_precision(tmp_path):
    path = tmp_path / "vae.ckpt"
    torch.save({"hyper_parameters": {"num_points": NP, "latent_dim": 256, "hidden_dim": 512}, "state_dict": _full_checkpoint()}, path)
    v = pcd_b200.SimplePointNetVAE.load_from_checkpoint(str(path), precision="f16mix")
    assert v.precision == "f16mix" and "precision" not in v.hparams
    assert torch.equal(v.fc_mu.weight, _full_checkpoint()["fc_mu.weight"])
    assert pcd_b200.SimplePointNetVAE.load_from_checkpoint(str(path)).precision == "bf16x3"


def test_oracle_transposes_clouds_to_channels_first():
    """The oracle's layout assumption, checked against torch's own modules: a [B, N, 3] cloud goes through the Conv1d stack as
    [B, 3, N], and AdaptiveMaxPool1d(1) + Flatten is the max over points."""
    full = _full_checkpoint()
    v = pcd_b200.SimplePointNetVAE(NP)
    v.load_state_dict(full, strict=True)
    v.eval()
    x = torch.randn(2, 77, 3, generator=torch.Generator().manual_seed(2))
    h = x.transpose(1, 2)
    with torch.no_grad():
        for i in range(4):
            layer = v.encoder[i]
            for j in (1, 2, 3):
                h = torch.relu(getattr(layer, f"bn{j}")(getattr(layer, f"conv{j}")(h)))
        h = v.encoder[7](v.encoder[6](v.encoder[5](v.encoder[4](h))))
        want = v.fc_mu(h), v.fc_logvar(h)
    mu, logvar = P.point_vae_encode({"vae." + k: t for k, t in full.items()}, x)
    assert torch.allclose(mu, want[0], rtol=1e-5, atol=1e-6) and torch.allclose(logvar, want[1], rtol=1e-5, atol=1e-6)


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference tree not mounted")
def test_encoder_oracle_vs_reference_module():
    _, rn, _ = ref_shim.load_reference()
    ref = rn.SimplePointNetVAE(NP)
    full = _full_checkpoint()
    ref.load_state_dict(full, strict=True)
    ref.eval()
    sd = {"vae." + k: t for k, t in full.items()}
    x = torch.randn(2, NP, 3, generator=torch.Generator().manual_seed(9))
    with torch.no_grad():
        mu, logvar = ref.encode(x)
        want_mu, want_lv = P.point_vae_encode(sd, x)
        assert torch.equal(mu, want_mu) and torch.equal(logvar, want_lv)
        torch.manual_seed(3)
        recon, fmu, flv = ref(x)
        torch.manual_seed(3)
        std = torch.exp(0.5 * want_lv)
        z = want_mu + torch.randn_like(std) * std
    assert torch.equal(fmu, want_mu) and torch.equal(flv, want_lv)
    assert torch.equal(recon, O.vae_decode(sd, z, NP))
